"""Truncated encode (cfbpe_encode_truncated): every prompt cut to a token budget, as fixed-length id rows, kept counts and the
byte cut of each prompt.  Expected results are the oracle's full encodings sliced in numpy; every cut is checked twice: as the
sum of the kept tokens' byte lengths (read from the rank file) and as the bytes the kept ids decode to.

The tests without a GPU run the window stage on the SIMT emulator (tests/simt/sim_truncate.cpp); the `gpu` ones run libcfbpe.so on the device."""
import base64
import os
import random

import numpy as np
import pytest

import fuzzgen
from conftest import COMBOS, pack

HEAD, TAIL = 0, 1
PAD = 0xFFFFFFF0
SLOT_NAMES = {0: "cl100k_base", 1: "o200k_base", 2: "llama3", 3: "tekken"}


@pytest.fixture(scope="module")
def token_bytes(tekken_bytes):
    """id -> the token's bytes (ids are ranks of the rank file; a slot of n ranks uses its first n lines)"""
    return [base64.b64decode(line.split()[0]) for line in tekken_bytes.splitlines()]


def check_window(token_bytes, prompts, ids, offs, counts, L, keep, budgets, rows, kept, got_counts, cut, n_decode=None):
    """rows / kept / counts / cut against the oracle's full encodings (ids, offs, counts), sliced in numpy.  Every cut is the sum of
    the kept tokens' byte lengths; for n_decode prompts (all by default) the kept ids also decode to exactly the cut's bytes."""
    n = len(prompts)
    tok_len = np.array([len(t) for t in token_bytes], dtype=np.uint64)
    c = np.asarray(counts, dtype=np.int64)
    k = np.minimum(c, L)
    if budgets is not None:
        k = np.minimum(k, np.asarray(budgets, dtype=np.int64))
    start = np.asarray(offs[:-1], dtype=np.int64) + (0 if keep == HEAD else c - k)      # first kept id of every prompt
    assert np.array_equal(got_counts, counts)
    assert np.array_equal(kept, k)
    if rows is not None and n:
        j = np.arange(L, dtype=np.int64)
        inside = j[None, :] < k[:, None]
        want_rows = np.where(inside, ids[np.minimum(start[:, None] + j[None, :], max(len(ids) - 1, 0))] if len(ids) else 0, PAD)
        bad = np.nonzero((rows != want_rows).any(axis=1))[0]
        assert not len(bad), (int(bad[0]), prompts[int(bad[0])][:80])
    if cut is None:
        return
    cum = np.zeros(len(ids) + 1, dtype=np.uint64)
    np.cumsum(tok_len[ids], out=cum[1:])
    nbytes = cum[start + k] - cum[start]
    plen = np.array([len(p) for p in prompts], dtype=np.uint64)
    want_cut = nbytes if keep == HEAD else plen - nbytes
    bad = np.nonzero(np.asarray(cut, dtype=np.uint64) != want_cut)[0]
    assert not len(bad), (int(bad[0]), int(cut[bad[0]]), int(want_cut[bad[0]]))
    pick = range(n) if n_decode is None else np.random.default_rng(n).choice(n, size=min(n, n_decode), replace=False)
    for i in pick:
        text = b"".join(token_bytes[t] for t in ids[start[i]:start[i] + k[i]])
        p, at = prompts[i], int(cut[i])
        assert (p[:at] if keep == HEAD else p[at:]) == text, (i, at)


def mixed_prompts(seed):
    """fuzz strings, long single-class runs (K2b / K2c pieces), runs of 1- to 3-byte prompts (many prompts in one flag word),
    empty prompts between non-empty ones, CJK and emoji (byte-level tokens: cuts inside characters)"""
    rng = random.Random(seed)
    out = [s.encode() for s in fuzzgen.fuzz_strings(seed, 300, max_atoms=40)] + [s.encode() for s in fuzzgen.long_runs(seed)[::3]]
    out += [b"", b"", b"a", b"", b"xy", b"", b"!!!"]
    out += [rng.choice([b"a", b"bc", b" d", b"\n", b"ef ", b"1"]) for _ in range(200)]
    out += [b"x" * 40, b"ab" * 150, b"abcdefgh" * 100, b" " * 700, b"7" * 300]
    out += ["中文日本語한글".encode() * 20, "\U0001f600\U0001f3f3️‍".encode() * 30, ("naïve café " * 30).encode(), b""]
    rng.shuffle(out)
    return out


def cuts_inside_characters(prompts, cut):
    """how many cuts fall inside a multi-byte UTF-8 character"""
    return sum(1 for p, c in zip(prompts, cut) if 0 < int(c) < len(p) and (p[int(c)] & 0xC0) == 0x80)


# ------------------------------------------------------------------ the emulator (no GPU)
@pytest.fixture(scope="module")
def sim_vocabs(tekken_bytes):
    import simtrunc
    return {pat: simtrunc.Vocab(tekken_bytes, 0, pat, n) for pat, n in COMBOS if pat in (0, 3)}


@pytest.fixture(scope="module")
def mixed(oracle_vocabs):
    from oracle import oracle
    prompts = mixed_prompts(17)
    data, offs = pack(prompts)
    ids, ioffs, counts = oracle.encode_batch([oracle_vocabs[0]], [0], data, offs)
    return prompts, ids, ioffs, counts


@pytest.mark.parametrize("keep", [HEAD, TAIL])
@pytest.mark.parametrize("L", [1, 2, 7, 64, 5000])
def test_window_on_emulator(sim_vocabs, token_bytes, mixed, keep, L):
    import simtrunc
    prompts, ids, ioffs, counts = mixed
    assert int(counts.max()) < 5000            # the largest L keeps every prompt whole
    rc, rows, kept, got_counts, cut, _ = simtrunc.encode_truncated([sim_vocabs[0]], prompts, L, keep, PAD)
    assert rc == 0
    check_window(token_bytes, prompts, ids, ioffs, counts, L, keep, None, rows, kept, got_counts, cut)
    if L <= 7:
        assert cuts_inside_characters(prompts, cut) > 0


@pytest.mark.parametrize("keep", [HEAD, TAIL])
def test_budgets_on_emulator(sim_vocabs, token_bytes, mixed, keep):
    import simtrunc
    prompts, ids, ioffs, counts = mixed
    rng = np.random.default_rng(5 + keep)
    budgets = rng.integers(0, 40, size=len(prompts)).astype(np.uint32)
    budgets[::7] = 0
    rc, rows, kept, got_counts, cut, _ = simtrunc.encode_truncated([sim_vocabs[0]], prompts, 24, keep, PAD, budgets=budgets)
    assert rc == 0
    check_window(token_bytes, prompts, ids, ioffs, counts, 24, keep, budgets, rows, kept, got_counts, cut)


@pytest.mark.parametrize("keep", [HEAD, TAIL])
def test_cuts_inside_long_and_big_pieces_on_emulator(sim_vocabs, oracle_vocabs, token_bytes, keep):
    """single pieces of 33..256 bytes (K2b) and above 256 bytes (K2c: ids by position), cut after every few tokens"""
    import simtrunc
    from oracle import oracle
    prompts = [b"ab" * 20, b"abcdefgh" * 30, b"a" * 257, b"xy" * 400, b"q" * 1000, ("中" * 200).encode()]
    data, offs = pack(prompts)
    ids, ioffs, counts = oracle.encode_batch([oracle_vocabs[3]], [3], data, offs)
    for L in (1, 3, 5, 11):
        rc, rows, kept, got_counts, cut, n_long = simtrunc.encode_truncated([sim_vocabs[3]], prompts, L, keep, PAD)
        assert rc == 0 and n_long > 0                                         # the long-piece kernels ran
        check_window(token_bytes, prompts, ids, ioffs, counts, L, keep, None, rows, kept, got_counts, cut)
        assert all(0 < int(c) < len(p) for p, c in zip(prompts, cut))       # every cut lies inside its (single-piece) prompt


def test_multi_vocabulary_batch_on_emulator(sim_vocabs, oracle_vocabs, token_bytes, mixed):
    import simtrunc
    from oracle import oracle
    prompts = mixed[0]
    vid = (np.arange(len(prompts)) % 2).astype(np.uint8)
    data, offs = pack(prompts)
    ids, ioffs, counts = oracle.encode_batch([oracle_vocabs[0], oracle_vocabs[3]], [0, 3], data, offs, vocab_ids=vid)
    for keep in (HEAD, TAIL):
        rc, rows, kept, got_counts, cut, _ = simtrunc.encode_truncated([sim_vocabs[0], sim_vocabs[3]], prompts, 9, keep, PAD, vocab_ids=vid)
        assert rc == 0
        check_window(token_bytes, prompts, ids, ioffs, counts, 9, keep, None, rows, kept, got_counts, cut)


def test_count_only_and_edge_batches_on_emulator(sim_vocabs, token_bytes, mixed):
    """rows = NULL (no id is written: the cut and kept counts alone), cut = NULL, a batch of empty prompts, an empty batch"""
    import simtrunc
    prompts, ids, ioffs, counts = mixed
    for keep in (HEAD, TAIL):
        rc, rows, kept, got_counts, cut, _ = simtrunc.encode_truncated([sim_vocabs[0]], prompts, 5, keep, PAD, want_rows=False)
        assert rc == 0 and rows is None
        check_window(token_bytes, prompts, ids, ioffs, counts, 5, keep, None, None, kept, got_counts, cut)
        rc, rows, kept, got_counts, cut, _ = simtrunc.encode_truncated([sim_vocabs[0]], prompts, 5, keep, PAD, want_cut=False)
        assert rc == 0 and cut is None
        check_window(token_bytes, prompts, ids, ioffs, counts, 5, keep, None, rows, kept, got_counts, None)
    rc, rows, kept, got_counts, cut, _ = simtrunc.encode_truncated([sim_vocabs[0]], [b"", b"", b""], 3, TAIL, PAD)
    assert rc == 0 and (kept == 0).all() and (got_counts == 0).all() and (cut == 0).all() and (rows == PAD).all()
    rc, rows, kept, got_counts, cut, _ = simtrunc.encode_truncated([sim_vocabs[0]], [], 3, HEAD, PAD)
    assert rc == 0 and len(kept) == 0


def test_malformed_utf8_on_emulator(sim_vocabs):
    import simtrunc
    rc = simtrunc.encode_truncated([sim_vocabs[0]], [b"fine", b"bad \xff", b"ok"], 4, HEAD, PAD)[0]
    assert rc != 0


# ------------------------------------------------------------------ the device
@pytest.fixture(scope="module")
def plug():
    from cfbpe import plugin as P
    p = P.GpuBpeTokenizerPlugin(device=0, vocab_names=("cl100k_base", "o200k_base", "llama3", "tekken"),
                                max_batch_bytes=256 << 20, max_prompts=1 << 17)
    yield p
    p.close()


@pytest.fixture(scope="module")
def sctx():
    from cfbpe import plugin as P
    return P.SecurityContext.anonymous()


def truncate(plug, sctx, name, data, offs, L, keep, budgets=None, want_ids=True, per_prompt=None):
    from cfbpe import plugin as P
    r = plug.truncate_batch(sctx, P.TruncateBatchRequest(P.VocabRef(name), data, offs, L, "head" if keep == HEAD else "tail", PAD,
                                                         budgets, want_ids, per_prompt))
    return r.rows, r.kept, r.counts, r.cut


@pytest.mark.gpu
@pytest.mark.parametrize("pat,n_ranks", COMBOS)
def test_fuzz_against_oracle_on_device(plug, sctx, oracle_vocabs, token_bytes, pat, n_ranks):
    from oracle import oracle
    prompts = mixed_prompts(900 + pat) + [s.encode() for s in fuzzgen.fuzz_strings(9100 + pat, 8000, max_atoms=48)]
    data, offs = pack(prompts)
    ids, ioffs, counts = oracle.encode_batch([oracle_vocabs[pat]], [pat], data, offs, nthreads=os.cpu_count())
    budgets = np.random.default_rng(pat).integers(0, 30, size=len(prompts)).astype(np.uint32)
    for keep in (HEAD, TAIL):
        for L, bud in ((1, None), (16, budgets), (4096, None)):
            got = truncate(plug, sctx, SLOT_NAMES[pat], data, offs, L, keep, bud)
            check_window(token_bytes, prompts, ids, ioffs, counts, L, keep, bud, *got)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_id", [3, 5])
def test_benchmark_configs_full_size_on_device(plug, sctx, token_bytes, cfg_id):
    """BASELINE.json configs 3 (65 536 prompts of 8..4096 B) and 5 (three vocabularies, per-prompt budgets) at full size"""
    from cfbpe import plugin as P
    from cfbpe import workload as W
    from oracle import oracle
    data, offs, vid, meta = W.make_config(cfg_id, 1.0)
    names = meta["vocabs"]
    ovs, pats = [], []
    for nm in names:
        rv = plug.resolved[nm]
        ovs.append(oracle.OracleVocab(rv.file_bytes, rv.max_ranks))
        pats.append(rv.pattern_id)
    ids, ioffs, counts = oracle.encode_batch(ovs, pats, data, offs, vocab_ids=vid if len(names) > 1 else None, nthreads=os.cpu_count())
    n = len(offs) - 1
    prompts = [bytes(data[int(offs[i]):int(offs[i + 1])]) for i in range(n)]
    per_prompt = [P.VocabRef(names[int(v)]) for v in vid] if len(names) > 1 else None
    budgets = np.random.default_rng(cfg_id).integers(0, 3000, size=n).astype(np.uint32) if cfg_id == 5 else None
    for L in (128, 4096):
        for keep in (HEAD, TAIL):
            got = truncate(plug, sctx, names[0], data, offs, L, keep, budgets, per_prompt=per_prompt)
            check_window(token_bytes, prompts, ids, ioffs, counts, L, keep, budgets, *got, n_decode=3000)


@pytest.mark.gpu
def test_pipelined_host_path_on_device(oracle_vocabs, tekken_bytes, token_bytes, monkeypatch):
    """the pipelined host path with tiny sub-batches (many seams, chained token ranks), empty prompts and a 30 000-byte prompt"""
    from cfbpe import _native as N
    from oracle import oracle
    monkeypatch.setenv("CFBPE_PIPE_CHUNK_BYTES", "20000")
    monkeypatch.setenv("CFBPE_PIPE_MIN_BYTES", "1")
    c = N.Context(0, 8 << 20, 1 << 15)
    c.vocab_load(0, tekken_bytes, N.FORMAT_TIKTOKEN, 0, 100256)
    c.vocab_load(1, tekken_bytes, N.FORMAT_TIKTOKEN, 1, 150000)
    prompts = [s.encode() for s in fuzzgen.fuzz_strings(4321, 12000, max_atoms=40) + fuzzgen.long_runs(8)] + [b"", b"", b"x" * 30000, b""]
    data, offs = pack(prompts)
    vid = (np.arange(len(prompts)) % 2).astype(np.uint8)
    ids, ioffs, counts = oracle.encode_batch([oracle_vocabs[0], oracle_vocabs[1]], [0, 1], data, offs, vocab_ids=vid, nthreads=os.cpu_count())
    budgets = np.random.default_rng(1).integers(0, 50, size=len(prompts)).astype(np.uint32)
    for keep in (HEAD, TAIL):
        for L, bud, want in ((8, budgets, True), (256, None, True), (512, None, False)):
            rows, kept, got_counts, cut = c.encode_truncated(data, offs, vid, max_tokens=L, keep=keep, pad_id=PAD, budgets=bud, want_ids=want)
            check_window(token_bytes, prompts, ids, ioffs, counts, L, keep, bud, rows, kept, got_counts, cut)
    bad = prompts[:3000] + [b"\xff\xfe"] + prompts[3000:6000]
    with pytest.raises(N.NativeError) as ei:
        c.encode_truncated(*pack(bad), max_tokens=4)
    assert ei.value.code == N.EILSEQ
    rows, kept, got_counts, cut = c.encode_truncated(data, offs, vid, max_tokens=8, keep=TAIL, pad_id=PAD)     # still healthy
    check_window(token_bytes, prompts, ids, ioffs, counts, 8, TAIL, None, rows, kept, got_counts, cut)
    c.close()


@pytest.mark.gpu
def test_device_entry_matches_host_entry(plug, oracle_vocabs):
    """cfbpe_encode_truncated_device on torch buffers and the current stream: two asynchronous calls back to back on reused
    buffers, then one status check; each equals the host entry"""
    import torch
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream().cuda_stream
    L = 64
    batches = []
    for seed, n in [(21, 5000), (22, 300)]:
        prompts = mixed_prompts(seed)[:n] + [s.encode() for s in fuzzgen.fuzz_strings(seed, n, max_atoms=60)]
        data, offs = pack(prompts)
        budgets = np.random.default_rng(seed).integers(0, 80, size=len(prompts)).astype(np.uint32)
        batches.append((data, offs, budgets))
    n_max = max(len(o) - 1 for _, o, _ in batches)
    total_max = max(len(d) for d, _, _ in batches)
    d_bytes = torch.zeros(total_max + 64, dtype=torch.uint8, device=dev)
    d_offs = torch.zeros(n_max + 1, dtype=torch.int64, device=dev)
    d_bud = torch.zeros(n_max, dtype=torch.int32, device=dev)
    outs = [dict(rows=torch.full((n_max, L), -1, dtype=torch.int32, device=dev), kept=torch.zeros(n_max, dtype=torch.int32, device=dev),
                 counts=torch.zeros(n_max, dtype=torch.int32, device=dev), cut=torch.zeros(n_max, dtype=torch.int64, device=dev))
            for _ in batches]
    for keep in (HEAD, TAIL):
        ins = []
        for (data, offs, budgets), o in zip(batches, outs):
            n, total = len(offs) - 1, len(data)
            ins.append((torch.from_numpy(np.concatenate([data, np.zeros(64, np.uint8)])).to(dev), torch.from_numpy(offs.astype(np.int64)).to(dev),
                        torch.from_numpy(budgets.view(np.int32)).to(dev)))
        for (data, offs, budgets), (b, of, bu), o in zip(batches, ins, outs):       # enqueue both without a sync in between
            n, total = len(offs) - 1, len(data)
            d_bytes[:total + 64].copy_(b); d_offs[:n + 1].copy_(of); d_bud[:n].copy_(bu)
            plug.ctx.encode_truncated_device(n, d_bytes.data_ptr(), total, d_offs.data_ptr(), None, L, keep, PAD, d_bud.data_ptr(),
                                             o["rows"].data_ptr(), o["kept"].data_ptr(), o["counts"].data_ptr(), o["cut"].data_ptr(), stream)
        plug.ctx.device_status(stream)
        for (data, offs, budgets), o in zip(batches, outs):
            n = len(offs) - 1
            rows, kept, counts, cut = plug.ctx.encode_truncated(data, offs, max_tokens=L, keep=keep, pad_id=PAD, budgets=budgets)
            assert np.array_equal(o["rows"][:n].cpu().numpy().view(np.uint32), rows)
            assert np.array_equal(o["kept"][:n].cpu().numpy().view(np.uint32), kept)
            assert np.array_equal(o["counts"][:n].cpu().numpy().view(np.uint32), counts)
            assert np.array_equal(o["cut"][:n].cpu().numpy().view(np.uint64), cut)


@pytest.mark.gpu
def test_error_codes_on_device(plug, sctx, tekken_bytes):
    from cfbpe import _native as N
    from cfbpe import plugin as P
    c = plug.ctx
    data, offs = pack([b"hello world", b"", b"more text here"])
    good = c.encode_truncated(data, offs, max_tokens=2)

    def code(d=data, o=offs, **kw):
        kw.setdefault("max_tokens", 2)
        with pytest.raises(N.NativeError) as ei:
            c.encode_truncated(d, o, **kw)
        return ei.value.code
    bad_d, bad_o = pack([b"ok", b"bad \xff"])
    assert code(max_tokens=0) == N.EINVAL
    assert code(keep=2) == N.EINVAL
    assert code(np.zeros(8, np.uint8), np.array([0, 5, 3, 8], dtype=np.uint64)) == N.EINVAL      # offsets not monotonic
    assert code(bad_d, bad_o) == N.EILSEQ
    assert code(vocab_ids=np.array([0, 7, 0], dtype=np.uint8)) == N.ENOENT
    lib = N.load()
    kept_buf, rows_buf = np.zeros(3, dtype=np.uint32), np.zeros(8, dtype=np.uint32)
    huge = plug.max_batch_bytes // 3 + 1            # 3 rows of it exceed max_batch_bytes: refused before anything is written
    assert lib.cfbpe_encode_truncated(c._h, 3, data.ctypes.data, offs.ctypes.data, None, huge, 0, 0, None, rows_buf.ctypes.data,
                                      kept_buf.ctypes.data, None, None) == N.EINVAL
    rows, kept, counts, cut = c.encode_truncated(data, offs, max_tokens=huge, want_ids=False)     # without rows there is no such limit
    assert np.array_equal(counts, good[2]) and np.array_equal(cut, [11, 0, 14])
    assert lib.cfbpe_encode_truncated(c._h, 3, data.ctypes.data, offs.ctypes.data, None, 2, 0, 0, None, None, None, None, None) == N.EINVAL
    assert lib.cfbpe_encode_truncated(c._h, 3, data.ctypes.data, offs.ctypes.data, None, 2, 0, 0, None, None, kept_buf.ctypes.data,
                                      None, None) == N.OK
    assert np.array_equal(kept_buf, good[1])
    with pytest.raises(P.InvalidInput):
        truncate(plug, sctx, "cl100k_base", *pack([b"bad \xff"]), 4, HEAD)
    with pytest.raises(P.VocabNotFound):
        truncate(plug, sctx, "no-such-vocab", data, offs, 4, HEAD)
    after = c.encode_truncated(data, offs, max_tokens=2)                  # the context still works
    assert all(np.array_equal(a, b) for a, b in zip(after, good))


@pytest.mark.gpu
def test_service_truncate_against_live_tiktoken(plug, sctx, tekken_bytes):
    """LlmGatewayTokenizerService.truncate on chat-sized texts against slices of live tiktoken encodings"""
    tiktoken = pytest.importorskip("tiktoken")
    from cfbpe import plugin as P
    from oracle import patterns as PT
    lines = tekken_bytes.splitlines()[:100256]
    enc = tiktoken.Encoding("live0", pat_str=PT.PATTERNS[0], mergeable_ranks={base64.b64decode(l.split()[0]): i for i, l in enumerate(lines)},
                            special_tokens={})
    hub = P.ClientHub()
    hub.register_scoped(P.TokenizerPluginClient, plug.instance.id, plug)
    svc = P.LlmGatewayTokenizerService(hub, [plug.instance])
    rng = random.Random(3)
    texts = ["".join(fuzzgen.fuzz_strings(rng.randint(0, 10 ** 6), 40, max_atoms=60)) for _ in range(200)]
    texts += ["You are a helpful assistant.  Summarise the following document:\n\n" + "Lorem ipsum dolor sit amet. " * 200,
              "中文日本語 " * 300, ""]
    for keep in ("head", "tail"):
        for L in (1, 50, 700):
            got = svc.truncate(sctx, "cl100k_base", texts, L, keep)
            for t, (ids, cut) in zip(texts, got):
                full = enc.encode_ordinary(t)
                want = full[:L] if keep == "head" else full[max(0, len(full) - L):]
                assert ids.tolist() == want
                b = t.encode()
                assert (b[:cut] if keep == "head" else b[cut:]) == enc.decode_bytes(want)


@pytest.mark.gpu
@pytest.mark.skipif("__import__('torch').cuda.device_count() < 2")
@pytest.mark.parametrize("mode", ["shards", "round_robin"])
def test_multi_device_truncation(oracle_vocabs, tekken_bytes, token_bytes, mode, monkeypatch):
    """a multi-device context returns exactly what one device returns: contiguous shards and round-robin sub-batches"""
    import torch
    from cfbpe import _native as N
    from oracle import oracle
    ndev = min(torch.cuda.device_count(), 8)
    if mode == "round_robin":
        monkeypatch.setenv("CFBPE_PIPE_MIN_BYTES", "1")
        monkeypatch.setenv("CFBPE_PIPE_CHUNK_BYTES", str(64 << 10))
    else:
        monkeypatch.setenv("CFBPE_NO_PEER", "1")
    prompts = [s.encode() for s in fuzzgen.fuzz_strings(78, 40000, max_atoms=60) + fuzzgen.long_runs(6)] + [b"", b"x", b""]
    data, offs = pack(prompts)
    vid = (np.arange(len(prompts)) % 2).astype(np.uint8)
    ids, ioffs, counts = oracle.encode_batch([oracle_vocabs[0], oracle_vocabs[3]], [0, 3], data, offs, vocab_ids=vid, nthreads=os.cpu_count())
    torch.cuda.set_device(0)
    c = N.Context(0, 64 << 20, 1 << 17, devices=list(range(ndev)))
    c.vocab_load(0, tekken_bytes, N.FORMAT_TIKTOKEN, 0, 100256)
    c.vocab_load(1, tekken_bytes, N.FORMAT_TIKTOKEN, 3, 130072)
    budgets = np.random.default_rng(2).integers(0, 40, size=len(prompts)).astype(np.uint32)
    for keep in (HEAD, TAIL):
        for L, bud in ((12, budgets), (300, None)):
            rows, kept, got_counts, cut = c.encode_truncated(data, offs, vid, max_tokens=L, keep=keep, pad_id=PAD, budgets=bud)
            check_window(token_bytes, prompts, ids, ioffs, counts, L, keep, bud, rows, kept, got_counts, cut)
    c.close()
    assert torch.cuda.current_device() == 0
