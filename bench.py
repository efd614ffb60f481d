#!/usr/bin/env python3
"""bench.py -- prompt-bytes/s of the batched BPE encode path (BASELINE.json metric).

  python bench.py [--gpus N --steps K --warmup W]         the CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference [...]                  the CPU implementation timed on the host cores
  python bench.py [...] --dump-outputs DIR                also write what the last timed step computed as DIR/<name>.npy

A "step" is one pass of the hot path over one synthetic batch: BASELINE.json configs[2]
(65 536 prompts, lengths uniform 8..4096 B, cl100k pattern) -- the config the north_star metric
is quoted on; it fits one GPU.  Weak scaling: every rank encodes its own 65 536-prompt shard
(seed 3 + rank), so the global batch is N x 65 536 prompts and there is no data-path collective;
the per-shard token totals are all_gathered every step (the path's only exchange).

  value     whole-job prompt-bytes/s, inputs resident in HBM (cfbpe_encode_batch_device on torch's stream)
  e2e       the same metric through the plugin / C ABI with pinned HOST buffers, H2D + D2H inside the timed region
  roofline  dominant kernel: algorithmic bytes / CUDA-event duration vs the measured HBM copy peak
  cpu_baseline  the oracle port on the host CPUs the container may use (cgroup quota), bounded sample, rank 0 only
  + extra records (the headline is unchanged by them): kernel_ms (CUDA events inside the library), parity (every rank's ids against
    the oracle), sustained (the device leg held ~2 s), strong / strong_one_context / config5 (the multi-GPU workloads BASELINE.json
    names), host_cpu (was the container's CPU quota hit during the e2e leg), numa, cpu_baseline_context (tiktoken's own batch call)
"""
import os
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA initialises: the pipelined host path keeps ~20 streams busy (DESIGN.md section 4)
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "cyberfabric-core_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "prompt_bytes_per_sec_bpe_encode"
UNIT = "bytes/s"
CONFIG_ID = 3
WORKLOAD = "BASELINE.json configs[2]: 65536 prompts/GPU, lengths uniform 8-4096 B (mix 80% english+code, 10% multilingual, " \
           "5% digits/whitespace, 5% adversarial), cl100k pattern"


def workload_config(rv, n_prompts, total_bytes, seed, scale):
    """what names the workload -- identical in the CUDA arm and the reference arm (the driver compares the two dicts);
    measured properties of the batch (tokens, long pieces ...) are reported under `workload_stats` instead"""
    return {"workload": WORKLOAD, "vocab": rv.label, "vocab_stand_in": rv.stand_in, "prompts_per_gpu": int(n_prompts),
            "total_bytes_per_gpu": int(total_bytes), "seed": int(seed), "scale": float(scale),
            "l2": "inputs (%.0f MB) and per-byte work arrays (> 1 GB) exceed the 126 MB L2; no flush needed" % (total_bytes / 1e6)}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the benchmark runs"""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_encode_rate(data, offs, rv, threads, target_s=12.0):
    """oracle port on `threads` host threads over a bounded prefix of the batch; returns (bytes/s, sample description)"""
    from oracle import oracle
    ov = oracle.OracleVocab(rv.file_bytes, rv.max_ranks)
    n = len(offs) - 1
    probe = min(n, 2048)

    def run(k):
        sub = offs[:k + 1]
        t0 = time.perf_counter()
        oracle.encode_batch([ov], [rv.pattern_id], data[:int(sub[-1])], sub, nthreads=threads, want_ids=True)
        return time.perf_counter() - t0, int(sub[-1])
    run(min(n, 256))                       # warm the tables
    t, b = run(probe)
    k = int(min(n, max(probe, probe * target_s / max(t, 1e-3))))
    t, b = run(k)
    return b / t, "first %d prompts (%d bytes) of the same batch, %.1f s wall" % (k, b, t), t, b


try:
    ALL_CPUS = os.sched_getaffinity(0)          # before any NUMA pinning
except Exception:
    ALL_CPUS = None


def host_cpu_budget():
    """How many host threads can really run: the CPUs of the affinity mask, capped by the cgroup CPU quota when there is one
    (a container that SEES 128 CPUs may be allowed far fewer; threads beyond the quota only get throttled).  -> (threads, facts)"""
    visible = os.cpu_count() or 1
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = visible
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max",):
        try:
            q, per = open(path).read().split()[:2]
            if q != "max":
                quota = float(q) / float(per)
        except Exception:
            pass
    if quota is None:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    n = aff if quota is None else max(1, min(aff, int(quota + 0.999)))
    return n, {"visible_cpus": visible, "affinity_cpus": aff, "cgroup_quota_cpus": quota}


def cgroup_throttle():
    """(nr_throttled, throttled_usec, usage_usec) of this container's CPU controller, or None"""
    try:
        kv = dict(l.split() for l in open("/sys/fs/cgroup/cpu.stat").read().splitlines())
        return int(kv.get("nr_throttled", 0)), int(kv.get("throttled_usec", 0)), int(kv.get("usage_usec", 0))
    except Exception:
        return None


def pin_to_gpu_numa_node(local_rank):
    """Run this rank -- and allocate its pinned buffers, which follow the allocating thread's node -- on the CPUs next to its GPU.
    With eight ranks the host leg is bound by the box's PCIe roots and memory: a rank whose buffers sit on the other socket pays
    the inter-socket link on every copy (SCALE_r01: e2e efficiency 0.87 at N = 8 without pinning).  Returns what was done."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1 and 64 * i + b < n_cpu]
        node = None
        try:
            node = int(pynvml.nvmlDeviceGetNumaNodeId(h))
        except Exception:
            pass
        if cpus and len(cpus) < n_cpu:
            os.sched_setaffinity(0, cpus)
            return {"pinned": True, "cpus": len(cpus), "first_cpu": cpus[0], "numa_node": node, "how": "nvml cpu affinity of the GPU"}
        return {"pinned": False, "why": "the GPU's affinity covers every CPU (one node, or not exposed here)", "numa_node": node}
    except Exception as e:   # noqa: BLE001
        return {"pinned": False, "why": "nvml affinity query failed: %s" % type(e).__name__}


def tiktoken_context_rate(data, offs, rv, threads, target_s=6.0):
    """context only (not the baseline of record): tiktoken 0.12.0 `encode_ordinary_batch(num_threads=threads)` on a prefix of the
    same batch, with the same ranks and pattern.  Returns a dict, or None when tiktoken is not importable."""
    try:
        import base64
        import tiktoken
        from oracle import patterns as PT
    except Exception:
        return None
    lines = rv.file_bytes.splitlines()
    if rv.max_ranks:
        lines = lines[:rv.max_ranks]
    ranks = {base64.b64decode(l.split()[0]): i for i, l in enumerate(lines) if l.strip()}
    enc = tiktoken.Encoding("bench", pat_str=PT.PATTERNS[rv.pattern_id], mergeable_ranks=ranks, special_tokens={})
    n = len(offs) - 1

    def run(k):
        texts = [bytes(data[int(offs[i]):int(offs[i + 1])]).decode("utf-8") for i in range(k)]
        t0 = time.perf_counter()
        enc.encode_ordinary_batch(texts, num_threads=threads)
        return time.perf_counter() - t0, int(offs[k])
    t, b = run(min(n, 512))
    k = int(min(n, max(512, 512 * target_s / max(t, 1e-3))))
    t, b = run(k)
    return {"value": b / t, "unit": UNIT, "cores": threads, "kind": "tiktoken 0.12.0 encode_ordinary_batch (python lists in and out)",
            "sample": "first %d prompts (%d bytes), %.1f s wall" % (k, b, t)}


DUMP_SEED = 20261017
DUMP_ID_BYTES = 15 << 20      # input bytes whose ids are written: a token covers at least one byte, so at most 60 MiB of ids


def dump_outputs(out_dir, offs, d_ids, d_out_off, d_counts):
    """Write what the device leg hands its caller, so that two builds can be compared output for output: the token offsets of
    every prompt (float64: they pass 2**24), the per-prompt token counts, and the ids of a fixed sample of prompts holding
    DUMP_ID_BYTES of input (ids stay below 2**24, exact in float32), with the sample's prompt indices.  The sample is drawn
    from the inputs alone, so equal inputs give equal samples whatever the build computes."""
    import torch
    n = len(offs) - 1
    out_off = d_out_off.cpu().numpy()
    order = np.random.default_rng(DUMP_SEED).permutation(n)
    in_bytes = np.cumsum(np.diff(offs.astype(np.int64))[order])
    pick = np.sort(order[:max(1, int(np.searchsorted(in_bytes, DUMP_ID_BYTES, side="right")))])
    pos = np.concatenate([np.arange(out_off[i], out_off[i + 1]) for i in pick])
    ids = d_ids[torch.from_numpy(pos).to(d_ids.device)].cpu().numpy().view(np.uint32)
    arrays = {"token_offsets": out_off.astype(np.float64), "token_counts": d_counts.cpu().numpy().astype(np.float32),
              "sample_prompts": pick.astype(np.float64), "sample_ids": ids.astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    """--impl reference: the CPU implementation on the host cores.  The reference tree has no tokenizer to
    compile (SURVEY.md F1), so this is the oracle port (oracle/bpe_oracle.c) on every host thread."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from cfbpe import vocabs as V
    from cfbpe import workload as W
    data, offs, vid, meta = W.make_config(CONFIG_ID, 1.0)
    rv = V.resolve("cl100k_base", allow_stand_in=True)
    threads, cpu_facts = host_cpu_budget()
    per_step = max(2.0, min(20.0, 120.0 / max(args.steps + args.warmup, 1)))
    for _ in range(args.warmup):
        cpu_encode_rate(data, offs, rv, threads, target_s=per_step / 2)
    tt = tb = 0.0
    sample = ""
    for _ in range(args.steps):
        rate, sample, t, b = cpu_encode_rate(data, offs, rv, threads, target_s=per_step)
        tt += t; tb += b
    value = tb / tt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": workload_config(rv, len(offs) - 1, meta["total_bytes"], W.CONFIGS[CONFIG_ID]["seed"], 1.0),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "each step: " + sample, "host": cpu_facts},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit_line(json.dumps(line))
    return 0


# stdout carries exactly ONE JSON line: libraries (NCCL prints its version there) get stderr instead
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit_line(text):
    os.write(_REAL_STDOUT, (text + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cfbpe", choices=["cfbpe", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the batch (debug only; a scaled run is not a bench value)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true", help="skip the extra config-5 record")
    ap.add_argument("--sustain-seconds", type=float, default=2.0, help="extra record: the device leg held this long (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps of the device leg, write what its last step "
                    "computed (rank 0's shard) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "cfbpe" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from cfbpe import _native as N
    from cfbpe import dist as D
    from cfbpe import plugin as P
    from cfbpe import workload as W

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            sys.stderr.write("bench.py: --gpus %d needs torchrun (one process per GPU)\n" % args.gpus)
            return 2
    numa = pin_to_gpu_numa_node(local_rank)      # before any pinned allocation
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    # ---- init: one rank parses the rank file, NCCL broadcasts the packed tables
    def factory(blobs):
        return P.GpuBpeTokenizerPlugin(device=local_rank, vocab_names=("cl100k_base",), max_batch_bytes=160 << 20,
                                       max_prompts=1 << 17, import_blobs=blobs, allow_stand_in=True)
    plug = D.load_vocab_everywhere(factory, ["cl100k_base"], 0, dev) if world > 1 else factory(None)
    rv = plug.resolved["cl100k_base"]
    ctx = P.SecurityContext.anonymous()

    # ---- this rank's shard (weak scaling: its own 64K-prompt batch)
    cfg = dict(W.CONFIGS[CONFIG_ID])
    n_prompts = max(1, int(round(cfg["n"] * args.scale)))
    data, offs, meta = W.make_batch(n_prompts, cfg["min_len"], cfg["max_len"], cfg["seed"] + rank)
    total = int(offs[-1])
    n = n_prompts

    # pinned host buffers for the e2e leg
    h_bytes = plug.ctx.pinned(total + 64, np.uint8); h_bytes.array[:total] = data
    h_offs = plug.ctx.pinned(n + 1, np.uint64); h_offs.array[:] = offs
    h_ids = plug.ctx.pinned(total + 1, np.uint32)
    h_out_off = plug.ctx.pinned(n + 1, np.uint64)
    h_counts = plug.ctx.pinned(n, np.uint32)
    # device-resident buffers for the kernel-only leg
    d_bytes = torch.zeros(total + 256, dtype=torch.uint8, device=dev)
    d_bytes[:total] = torch.from_numpy(data).to(dev)
    d_offs = torch.from_numpy(offs.astype(np.int64)).to(dev)
    d_ids = torch.empty(total + 1, dtype=torch.int32, device=dev)
    d_out_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    d_counts = torch.empty(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    totals = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]

    def step_device():
        plug.ctx.encode_batch_device(n, d_bytes.data_ptr(), total, d_offs.data_ptr(), None, d_ids.data_ptr(), d_ids.numel(),
                                     d_out_off.data_ptr(), d_counts.data_ptr(), stream, sync=False)
        if world > 1:
            dist.all_gather(totals, d_out_off[n:n + 1])

    def step_e2e():
        req = P.EncodeBatchRequest(P.VocabRef("cl100k_base"), h_bytes.array[:total], h_offs.array)
        return plug.encode_batch(ctx, req, out=P.EncodeBatchResponse(h_ids.array, h_out_off.array, h_counts.array))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # clocks and throttle reasons are sampled (every 50 ms) from the first warm-up step to the last end-to-end step: the GPU
    # is under this benchmark's load the whole time, and the timed regions alone (tens of ms) are shorter than nvidia-smi's start-up
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- kernel-only leg (inputs resident in HBM)
    for _ in range(args.warmup):
        step_device()
    barrier()
    plug.ctx.device_status(stream)          # warm-up result sanity: raises on bad UTF-8
    n_tokens = int(d_out_off[n].item())
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_device()
    e1.record()
    barrier()
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    total_all = sum_over_ranks(float(total))
    tokens_all = sum_over_ranks(float(n_tokens))
    value = total_all * args.steps / (dev_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, offs, d_ids, d_out_off, d_counts)

    # ---- the same leg held for ~2 s (the K timed steps above are tens of milliseconds): a sustained rate under sustained clocks
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / max(dev_ms / args.steps, 1e-3)))
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(n_sus):
            step_device()
        s1.record()
        barrier()
        sus_ms = max_over_ranks(s0.elapsed_time(s1))
        plug.ctx.device_status(stream)
        sustained = {"steps": n_sus, "seconds": sus_ms / 1e3, "ms_per_step": sus_ms / n_sus, "value": total_all * n_sus / (sus_ms * 1e-3), "unit": UNIT}

    # ---- per-kernel device times (CUDA events inside the library, same stream), averaged over the steps
    plug.ctx.profile_enable(True)
    kms = {k: 0.0 for k in N.KERNEL_NAMES}
    for _ in range(args.steps):
        plug.ctx.encode_batch_device(n, d_bytes.data_ptr(), total, d_offs.data_ptr(), None, d_ids.data_ptr(), d_ids.numel(),
                                     d_out_off.data_ptr(), d_counts.data_ptr(), stream, sync=True)
        pr = plug.ctx.profile_read()
        for k in N.KERNEL_NAMES:
            kms[k] += pr["kernel_ms"][k] / args.steps
    n_long = pr["n_long_pieces"]
    long_bytes, long_tokens = pr["n_long_bytes"], pr["n_long_tokens"]
    plug.ctx.profile_enable(False)

    # ---- end-to-end leg: pinned host buffers through the plugin / C ABI, H2D and D2H inside the timed region
    for _ in range(args.warmup):
        r = step_e2e()
    barrier()
    thr0 = cgroup_throttle()
    t0 = time.perf_counter()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(args.steps):
        r = step_e2e()
    c1.record()
    barrier()
    e2e_ms = max_over_ranks(max(c0.elapsed_time(c1), (time.perf_counter() - t0) * 1e3))
    e2e_value = total_all * args.steps / (e2e_ms * 1e-3)
    thr1 = cgroup_throttle()
    # was the container's CPU quota hit while the host legs of all ranks ran?  (each rank enqueues ~350 launches a step and waits
    # on events; a throttled rank stalls its pipeline.)  Container-wide counters, read by rank 0.
    host_cpu = None if thr0 is None or thr1 is None else {
        "cgroup_quota_cpus": host_cpu_budget()[1]["cgroup_quota_cpus"], "throttled_periods_during_e2e": thr1[0] - thr0[0],
        "throttled_ms_during_e2e": (thr1[1] - thr0[1]) / 1e3, "cpu_ms_used_during_e2e": (thr1[2] - thr0[2]) / 1e3, "wall_ms": e2e_ms}
    assert int(r.offsets[n]) == n_tokens
    # ---- the two multi-GPU workloads BASELINE.json names, as extra records (the headline stays the weak-scaled config 3):
    #   strong   configs[2] as ONE 65 536-prompt batch sharded by bytes over the N ranks (cfbpe.dist.shard_by_bytes); timed end to
    #            end from host buffers, the host-side sharding and the gather of the per-prompt counts inside the timed region
    #   config5  configs[4]: 256 tenants x 256 prompts, vocabulary = tenant mod 3 (cl100k / o200k / llama3 patterns), sharded likewise
    def sharded_leg(g_data, g_offs, g_vid, names):
        # The request buffers are pinned host memory, as in the e2e leg (set-up, untimed): the whole batch once; a shard is a
        # VIEW of it (no copy), its offsets rebased on the host inside the timed region.
        table = [P.VocabRef(nm) for nm in names]
        g_pin = plug.ctx.pinned(len(g_data) + 64, np.uint8)
        g_pin.array[:len(g_data)] = g_data
        g_view = g_pin.array[:len(g_data)]
        stage = {"g": g_pin}

        def once():
            sh_bytes, sh_offs, sh_vid, (lo, hi) = D.shard_batch(g_view, g_offs, g_vid, rank, world)     # host-side sharding: inside the timed region
            nb, nn = int(sh_offs[-1]), len(sh_offs) - 1
            if "hi" not in stage:                                           # pinned output buffers of this rank's shard, allocated once
                stage["hi"] = plug.ctx.pinned(nb + 1, np.uint32); stage["hoo"] = plug.ctx.pinned(nn + 1, np.uint64); stage["hc"] = plug.ctx.pinned(max(nn, 1), np.uint32)
            req = P.EncodeBatchRequest(table[0], sh_bytes, sh_offs, None if sh_vid is None else table, None if sh_vid is None else sh_vid)
            res = plug.encode_batch(ctx, req, out=P.EncodeBatchResponse(stage["hi"].array, stage["hoo"].array, stage["hc"].array))
            # the path's exchange: per-prompt counts of every shard (every rank cut the batch the same way and knows the sizes)
            counts = D.gather_counts(res.counts, dev, sizes=[h - l for l, h in D.shard_by_bytes(g_offs, world)]) if world > 1 else res.counts
            return res, counts, (lo, hi), nb
        for _ in range(args.warmup):
            once()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res, counts, span, nb = once()
        barrier()
        ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        return res, counts, span, nb, ms

    strong = None
    s_data, s_offs, _, s_meta = (data, offs, None, None) if rank == 0 and args.scale == 1.0 else W.make_config(CONFIG_ID, args.scale)[:4]
    res, counts, span, nb, ms = sharded_leg(s_data, s_offs, None, ["cl100k_base"])
    strong = {"workload": "configs[2] as ONE batch of %d prompts (%d bytes) sharded by bytes over %d GPU(s)" % (len(s_offs) - 1, int(s_offs[-1]), world),
              "value": int(s_offs[-1]) * args.steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / args.steps, "shard_bytes_rank0": nb,
              "tokens_total": int(np.asarray(counts, dtype=np.int64).sum()),
              "timed": "host sharding + H2D + kernels + D2H + gather of per-prompt counts (wall clock, max over ranks)"}
    # the same batch through ONE context over all the GPUs of the run (cfbpe_config.devices[]): sharding, the NCCL gather of
    # the totals and the rebasing of the offsets happen inside the library; rank 0 makes the call, the other ranks wait
    strong_lib = None
    if world > 1:
        # the other ranks wait on the CPU (a gloo barrier): an NCCL barrier would keep a spinning kernel on every GPU this context uses
        cpu_group = dist.new_group(backend="gloo")
        barrier()
        if rank == 0:
            try:
                from cfbpe import _native as NN
                cN = NN.Context(0, int(s_offs[-1]) + 4096, len(s_offs), devices=list(range(world)))     # every device can hold the batch: sub-batches go round-robin
                cN.vocab_load(0, rv.file_bytes, rv.spec.fmt, rv.pattern_id, rv.max_ranks or 0)
                hb = cN.pinned(len(s_data) + 64, np.uint8); hb.array[:len(s_data)] = s_data
                ho = (cN.pinned(int(s_offs[-1]) + 1, np.uint32), cN.pinned(len(s_offs), np.uint64), cN.pinned(len(s_offs), np.uint32))
                for _ in range(args.warmup):
                    rN = cN.encode_batch(hb.array[:len(s_data)], s_offs, None, *[x.array for x in ho])
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    rN = cN.encode_batch(hb.array[:len(s_data)], s_offs, None, *[x.array for x in ho])
                msN = (time.perf_counter() - t0) * 1e3
                same = bool(int(rN[1][-1]) == int(np.asarray(counts, dtype=np.int64).sum()) and np.array_equal(rN[2], np.asarray(counts, dtype=np.uint32)))
                strong_lib = {"workload": "the same batch through ONE context over %d devices (cfbpe_config.devices[]), one host process: the sub-batches of "
                                          "the pipelined call go round-robin over the devices, token ranks chained over NVLink peer memory" % world,
                              "value": int(s_offs[-1]) * args.steps / (msN * 1e-3), "unit": UNIT, "ms_per_step": msN / args.steps,
                              "counts_equal_to_the_sharded_leg": same}
                cN.close()
            except Exception as e:   # noqa: BLE001
                strong_lib = {"error": "%s: %s" % (type(e).__name__, e)}
        dist.barrier(group=cpu_group)
        torch.cuda.set_device(dev)
        barrier()
    config5 = None
    if not args.no_config5:
        c_data, c_offs, c_vid, c_meta = W.make_config(5, args.scale)
        for nm in c_meta["vocabs"]:
            if nm not in plug._slot:      # rank 0 parses, the packed tables travel by NCCL broadcast (cfbpe.dist)
                if world == 1:
                    plug.load_vocab(nm)
                elif rank == 0:
                    plug.load_vocab(nm); D.broadcast_blob(plug.export_vocab(nm), 0, dev)
                else:
                    plug.load_vocab(nm, D.broadcast_blob(None, 0, dev))
        res5, counts5, span5, nb5, ms5 = sharded_leg(c_data, c_offs, c_vid, c_meta["vocabs"])
        ok5 = True
        if rank == 0:      # a sample of rank 0's shard against the oracle (checker only, untimed)
            from oracle import oracle as _o
            ovs = [_o.OracleVocab(plug.resolved[nm].file_bytes, plug.resolved[nm].max_ranks) for nm in c_meta["vocabs"]]
            pats = [plug.resolved[nm].pattern_id for nm in c_meta["vocabs"]]
            for i in np.random.default_rng(5).choice(span5[1] - span5[0], size=min(256, span5[1] - span5[0]), replace=False):
                g = span5[0] + int(i); v = int(c_vid[g])
                want = ovs[v].encode(pats[v], bytes(c_data[int(c_offs[g]):int(c_offs[g + 1])]))
                ok5 = ok5 and np.array_equal(res5.ids[int(res5.offsets[i]):int(res5.offsets[i + 1])], want)
        config5 = {"workload": "configs[4]: %d tenants x %d prompts, vocabulary = tenant mod 3 (%s), %d bytes, sharded by bytes over %d GPU(s)"
                               % (256, (len(c_offs) - 1) // 256, "/".join(c_meta["vocabs"]), int(c_offs[-1]), world),
                   "value": int(c_offs[-1]) * args.steps / (ms5 * 1e-3), "unit": UNIT, "ms_per_step": ms5 / args.steps,
                   "tokens_total": int(np.asarray(counts5, dtype=np.int64).sum()), "parity_sample_rank0_ok": bool(ok5),
                   "vocab_stand_in": True}
    clocks = sampler.stop() if rank == 0 else None
    # ---- parity of what was just timed, on EVERY rank (ranks != 0 run on NCCL-broadcast tables): each rank hashes its id stream and
    #      hands rank 0 a seeded sample of its prompts with the ids the e2e leg produced and the ids the device leg left in HBM;
    #      rank 0 encodes the samples with the oracle (checker only, outside the timed regions) and compares
    import hashlib
    dev_ids = d_ids[:n_tokens].cpu().numpy().view(np.uint32)
    dev_off = d_out_off.cpu().numpy().astype(np.uint64)
    same_legs = bool(np.array_equal(dev_ids, r.ids[:n_tokens]) and np.array_equal(dev_off, r.offsets))
    pick = np.sort(np.random.default_rng(1000 + rank).choice(n, size=min(n, 512), replace=False))
    mine = {"rank": rank, "ids_sha256": hashlib.sha256(dev_ids.tobytes()).hexdigest()[:16], "n_tokens": n_tokens, "same_legs": same_legs,
            "prompts": [bytes(data[int(offs[i]):int(offs[i + 1])]) for i in pick],
            "ids": [dev_ids[int(dev_off[i]):int(dev_off[i + 1])].copy() for i in pick]}
    gathered = [mine]
    if world > 1:
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(mine, gathered, dst=0)
    h2d = total + (n + 1) * 8
    d2h = n_tokens * 4 + (n + 1) * 8 + n * 4 + 24

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    from oracle import oracle
    ov = oracle.OracleVocab(rv.file_bytes, rv.max_ranks)
    ok_ranks, bad = 0, []
    for g in gathered:
        good = g["same_legs"] and all(np.array_equal(ov.encode(rv.pattern_id, p), i) for p, i in zip(g["prompts"], g["ids"]))
        ok_ranks += 1 if good else 0
        if not good:
            bad.append(g["rank"])
    parity = {"parity_checked_ranks": ok_ranks, "ranks": world, "prompts_per_rank": len(gathered[0]["prompts"]),
              "checker": "oracle port, per-prompt ids; device leg == e2e leg on every rank", "mismatching_ranks": bad,
              "ids_sha256_per_rank": [g["ids_sha256"] for g in gathered]}
    if bad:
        sys.stderr.write("bench.py: PARITY FAILURE on ranks %s\n" % bad)
        return 3

    # ---- roofline of the dominant kernel
    hbm_gbs, peak_src = peaks()
    n_miss, n_list, list_parts = pr["n_miss_pieces"], pr["n_list_pieces"], pr["n_list_parts"]
    list_bytes = min(list_parts, long_bytes)      # bpe_list starts from the bytes: its parts at the start are its bytes
    n_extra = pr["n_extra_tokens"]
    n_pieces = (n_tokens - long_tokens) - n_extra + n_miss + n_long        # every short piece is one token or a miss; long pieces once
    alg = {  # algorithmic bytes per launch (DESIGN.md section 4)
        "pretok_split": total * (1 + 1 / 8 + 1 / 8) + 12 * (n + 1),              # text in, prompt-start flags in, piece-start flags out; offsets
        "long_scan": total / 8 + 24.0 * n_long + 4 * total / 2048,                # flags in; work-list entries and per-tile piece counts out
        "bpe_encode": total * (1 + 1 / 8) + 4.0 * n_pieces + total / 8 + 8.0 * n_miss + 12 * total / 2048,   # text + flags in; one word per piece, id flags, miss lists out
        "bpe_merge": n_miss * (8 + 8 + 4) + 4.0 * n_extra,                        # list entry, ~8 piece bytes, the piece's word; its tokens
        # the long pieces are shared by two kernels: bpe_list takes the ones above 256 bytes FROM THEIR BYTES (list_bytes of them;
        # their ids are apportioned by bytes: the status block counts the ids of both kernels together), bpe_long the rest
        "bpe_long": (long_bytes - list_bytes) * (1 + 4.0 * long_tokens / max(long_bytes, 1)) + 24.0 * (n_long - n_list),
        "bpe_list": list_bytes * (1 + 4.0 * long_tokens / max(long_bytes, 1)) + 24.0 * n_list,
        "flag_count": 3 * total / 8,                                             # token flags in, piece flags in, token flags out (ORed)
        "tile_scan": 0.0,
        "emit_compact": 2 * total / 8 + 4.0 * n_pieces + 4.0 * n_extra + 4.0 * long_tokens + 4.0 * n_tokens + 12 * (n + 1),   # both flag arrays, ids by piece, extras, long ids; ids out
        "reserved": 0.0,
    }
    dom = max(kms, key=lambda k: kms[k])
    achieved = alg[dom] / (kms[dom] * 1e-3) / 1e9 if kms[dom] > 0 else 0.0
    # dram bytes of that kernel from the committed `ncu --set full` capture -- only if the capture is of THIS build of the kernels
    traffic, traffic_note = None, "no ncu capture committed for this build"
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if tj.get("build_id") == N.load().cfbpe_build_id().decode():
                traffic, traffic_note = tj.get(dom), "profiles/ncu_traffic.json (build %s)" % tj.get("build_id")
            else:
                traffic_note = "profiles/ncu_traffic.json is of build %s, this is %s: stale, not reported" % (tj.get("build_id"), N.load().cfbpe_build_id().decode())
        except Exception:
            traffic = None
    path_alg = total + 4 * n_tokens + 21 * n
    kernels_ms = sum(kms.values())

    cpu, cpu_ctx = None, None
    if not args.no_cpu_baseline:
        mask = os.sched_getaffinity(0)
        try:                                      # the CPU legs get every host CPU, not only the ones next to the GPU
            os.sched_setaffinity(0, ALL_CPUS or mask)
        except Exception:
            pass
        threads, cpu_facts = host_cpu_budget()
        rate, sample, _, _ = cpu_encode_rate(data, offs, rv, threads)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "host": cpu_facts}
        cpu_ctx = tiktoken_context_rate(data, offs, rv, threads)
        os.sched_setaffinity(0, mask)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": workload_config(rv, n, total, cfg["seed"], args.scale),
        "parallelism": "dp%d (batch-sharded, no data-path collective; rank r encodes the batch of seed %d + r)" % (world, cfg["seed"]),
        "workload_stats": {"tokens_per_gpu": n_tokens, "bytes_per_token": total / max(n_tokens, 1), "long_pieces_per_gpu": int(n_long),
                           "long_piece_bytes_per_gpu": int(long_bytes), "short_miss_pieces_per_gpu": int(n_miss),
                           "list_pieces_per_gpu": int(n_list), "list_parts_per_gpu": int(list_parts)},
        "parity": parity,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms / args.steps, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": 13 * args.steps,   # prompt map, split, split fix-up, long-piece scan, big pieces (list), long pieces, piece-rank scan, piece lookup, short-piece merges, flag_count, tile_scan, emit, offsets
        "kernel_ms": kms,   # CUDA-event durations; bpe_long runs on a second stream next to bpe_encode, so they overlap
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s", "frac": achieved / hbm_gbs,
                     "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg[dom],
                     "path_algorithmic_bytes": path_alg,
                     "path_achieved_gbs": path_alg / (kernels_ms * 1e-3) / 1e9 if kernels_ms > 0 else 0.0},
        "strong": strong, "strong_one_context": strong_lib, "host_cpu": host_cpu, "sustained": sustained,
        "config5": config5,
        "numa": numa,
        "cpu_baseline": cpu,
        "cpu_baseline_context": cpu_ctx,
        "clocks": clocks,
    }
    emit_line(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
