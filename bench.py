#!/usr/bin/env python3
"""bench.py -- one JSON line per run (see the driver contract in the task statement).

Workload (BASELINE.json configs[4], the one `metric` is quoted on): a synthetic NDJSON
stream of parking-citations-shaped records (tests/golden/data/parking-citations.json.zst
replicated; no RNG).  A *step* is one pass of the hot path -- stage 1 + flatten, then the
stage-2 tape build -- over one batch of `--batch-mib` MiB on each GPU (weak scaling:
every rank parses its own shard of the stream; record boundaries are shard boundaries).

  value     GB/s of JSON parsed, whole job, inputs already resident in HBM, outputs left in
            HBM (sj_parse_device through the C ABI), timed with CUDA events on the
            library's stream, max over ranks
  e2e       same metric through the reference-facing call sj_parse() with HOST buffers:
            pinned host input -> H2D -> K1..K2f -> D2H of tape + strings, every step
  roofline  stage1_flatten kernel alone on the same batch: algorithmic bytes
            (N_in + 4 * N_idx, SURVEY.md 8d) / CUDA-event time, against the measured HBM peak
  cpu_baseline / --impl reference
            the reference cannot be built here (no Go toolchain), so the CPU arm is the
            oracle port (C restatement; AVX-512BW mask routines when the host has them, else AVX2+PCLMUL) run
            ParseNDStream-style on all host threads (10 MiB newline-aligned chunks)

--dump-outputs DIR writes what the last timed step of `value` left in HBM, i.e. what a caller of sj_parse_device
receives, so that two builds can be compared output for output on the same (deterministic) batch:
  tape.npy      float64 [k, 2]: high and low 32-bit halves of k tape words (exact in float64)
  strings.npy   float32 [k]: k bytes of the string buffer
  sizes.npy     float64 [2]: tape words, string bytes
k = min(length, 2^21 / ranks); when the output is longer, one position per equal stratum at a seeded offset (a
fixed sample for a given length).  With N > 1 every rank writes its slice as <name>_rank<r>.npy.  40 MiB of data at most.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True  # the benchmark leaves the tree as build() left it (it may be read-only)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "simdjson-go_b200"))

import numpy as np  # noqa: E402

# BASELINE.json's metric, verbatim, in BOTH arms (the driver matches the two lines on it)
METRIC = "GB/s JSON parsed end-to-end; stage1 achieved HBM GB/s vs B200 peak"
WORKLOAD = ("synthetic NDJSON stream: parking-citations-shaped records (BASELINE configs[4]), ParseND, copy_strings=true")


def load_records():
    from tests.util import load_fixture
    return load_fixture("parking-citations").strip()


def make_batch(nbytes):
    """NDJSON batch of about nbytes: the 1000-record fixture repeated, newline separated."""
    blk = load_records() + b"\n"
    k = max(1, nbytes // len(blk))
    buf = (blk * k)[:-1]  # no trailing newline: the parse trims anyway
    return buf


def host_threads():
    """threads for the CPU arm: the logical CPUs this process may use, capped by a cgroup quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = ""
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, period = f.read().split()
        quota = "cpu.max=%s/%s" % (q, period)
        if q != "max":
            n = max(1, min(n, -(-int(q) // int(period))))
    except Exception:
        pass
    return n, quota


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.samples = []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------
# CPU arm: the oracle port, ParseNDStream-shaped (simdjson_amd64.go:116-215)
# --------------------------------------------------------------------------------------
_cpu_pool = None
_cpu_isa = "?"
_cpu_local = threading.local()


def cpu_parse_stream(buf, threads, chunk=10 << 20, count_where=None):
    """Parse `buf` as NDJSON in newline-aligned ~10 MiB chunks on `threads` host threads
    (persistent workers with reused output buffers, like the reference's `reuse` channel,
    simdjson_amd64.go:116).  With count_where=(key, value) every chunk's tape is then walked by
    countWhere (ndjson_test.go:421).  Returns (seconds, bytes parsed)."""
    global _cpu_pool
    from concurrent.futures import ThreadPoolExecutor
    from oracle.pyoracle import FLAG_COPY_STRINGS, FLAG_NDJSON, Oracle
    o = Oracle("best")  # AVX-512BW mask routines when the host has them (the reference's choice, stage1_find_marks_amd64.go:42), else AVX2
    global _cpu_isa
    _cpu_isa = o.isa
    if _cpu_pool is None or _cpu_pool._max_workers != threads:
        _cpu_pool = ThreadPoolExecutor(max_workers=threads)
    arr = np.frombuffer(buf, dtype=np.uint8)
    cuts = [0]
    while cuts[-1] < len(buf):
        nxt = cuts[-1] + chunk
        if nxt >= len(buf):
            cuts.append(len(buf))
            break
        j = buf.find(b"\n", nxt)
        cuts.append(len(buf) if j < 0 else j + 1)
    local = _cpu_local

    def work(i):
        a, b = cuts[i], cuts[i + 1]
        n = b - a
        if not hasattr(local, "tape") or local.cap < n:
            local.cap = n + (n >> 2)
            local.tape = np.empty(2 * local.cap + 64, dtype=np.uint64)
            local.strs = np.empty(local.cap + 64, dtype=np.uint8)
        tl, sl, mo, ml = C.c_size_t(0), C.c_size_t(0), C.c_size_t(0), C.c_size_t(0)
        rc = o.lib.sjo_parse(arr[a:b].ctypes.data, n, FLAG_NDJSON | FLAG_COPY_STRINGS, local.tape.ctypes.data,
                             local.tape.size, C.byref(tl), local.strs.ctypes.data, local.strs.size, C.byref(sl),
                             C.byref(mo), C.byref(ml))
        assert rc == 0, rc
        if count_where:
            roots = C.c_uint64(0)
            o.lib.sjo_count_where(local.tape.ctypes.data, tl.value, local.strs.ctypes.data, arr[a + mo.value:].ctypes.data,
                                  count_where[0], len(count_where[0]), count_where[1], len(count_where[1]), C.byref(roots))
        return n

    t0 = time.perf_counter()
    total = sum(_cpu_pool.map(work, range(len(cuts) - 1)))
    return time.perf_counter() - t0, total


def run_reference(args, rank, world):
    """--impl reference: the CPU implementation of the path on the box's host cores."""
    if rank != 0:
        return
    threads, quota = host_threads()
    sample = make_batch(max(args.batch_mib, 1024) << 20)  # >= 100 chunks of 10 MiB so every host thread has work
    warm = sample[: 64 << 20]
    warm = warm[: warm.rfind(b"\n")]
    for _ in range(args.warmup):
        cpu_parse_stream(warm, threads)
    cpu_parse_stream(sample, threads)  # first touch of every worker's buffers stays outside the timed steps
    secs = 0.0
    nbytes = 0
    for _ in range(args.steps):
        t, n = cpu_parse_stream(sample, threads)
        secs += t
        nbytes += n
    gbs = nbytes / secs / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": round(gbs, 4),
        "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(secs / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "cpu_arm": "ParseNDStream-style 10 MiB newline-aligned chunks on all host threads",
                   "batch_bytes": len(sample)},
        "cpu_baseline": {"value": round(gbs, 4), "unit": "GB/s", "cores": threads, "kind": "port",
                         "isa": _cpu_isa,
                         "sample": "%d MiB per step, oracle port (C restatement of the reference's path, %s mask routines; the Go reference cannot be built: no Go toolchain) %s" % (len(sample) >> 20, _cpu_isa, quota)},
        "e2e": {"value": round(gbs, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def k1_traffic(batch_bytes):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE K1 launch on this batch, from the committed
    `ncu --set full` capture of this very command (profiles/k1_traffic.json); None for other batch sizes."""
    try:
        with open(os.path.join(ROOT, "profiles", "k1_traffic.json")) as f:
            t = json.load(f)
        return t["dram_bytes_read"] + t["dram_bytes_write"] if int(t["batch_bytes"]) == int(batch_bytes) else None
    except (OSError, ValueError, KeyError):
        return None


DUMP_SAMPLES = 1 << 21


def sample_index(length, k, seed):
    """k increasing positions in [0, length): every position when length <= k, else one per stratum of
    length // k or more positions, at a seeded offset inside it"""
    if length <= k:
        return np.arange(length, dtype=np.int64)
    rng = np.random.default_rng(seed)
    return np.arange(k, dtype=np.int64) * length // k + rng.integers(0, length // k, k)


def dump_outputs(out_dir, suffix, k, d_tape, tape_words, d_strings, string_bytes):
    """--dump-outputs: a fixed sample of the tape and string buffer in device memory (see the module docstring)"""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    ti = torch.from_numpy(sample_index(tape_words, k, 1)).to(d_tape.device)
    words = d_tape[ti].cpu().numpy().view(np.uint64)
    si = torch.from_numpy(sample_index(string_bytes, k, 2)).to(d_strings.device)
    sbytes = d_strings[si].cpu().numpy()
    halves = np.stack([words >> np.uint64(32), words & np.uint64(0xFFFFFFFF)], axis=1)
    np.save(os.path.join(out_dir, "tape%s.npy" % suffix), halves.astype(np.float64))
    np.save(os.path.join(out_dir, "strings%s.npy" % suffix), sbytes.astype(np.float32))
    np.save(os.path.join(out_dir, "sizes%s.npy" % suffix), np.array([tape_words, string_bytes], dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-mib", type=int, default=512, help="NDJSON bytes per step per GPU")
    ap.add_argument("--cpu-sample-mib", type=int, default=1024)
    ap.add_argument("--inflight", type=int, default=3, help="host-API calls kept in flight for the e2e number")
    ap.add_argument("--twitter-mib", type=int, default=1024, help="size of the twitter.json-shaped document of roofline_twitter (0: skip)")
    ap.add_argument("--stream-gib", type=int, default=64, help="GiB pushed through sj_stream_* per GPU-SET (split over the ranks); 0: skip")
    ap.add_argument("--stream-ring-mib", type=int, default=1024, help="size of the pinned ring of generated records each rank cycles over")
    ap.add_argument("--stream-chunk-mib", type=int, default=256, help="chunk size of the library's stream pipeline")
    ap.add_argument("--nccl-exchange", action="store_true", help="N > 1: exchange the shard totals through NCCL even where the peer-memory kernel is available (A/B)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's tape and strings to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import simdjson_b200 as sj
    from simdjson_b200 import _lib

    if not torch.cuda.is_available() or not sj.SupportedCPU():
        raise SystemExit("bench.py: no CUDA sm_100 device -- the CUDA path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    ctx = sj.Context(local_rank)
    L = ctx.L
    # host threads and pinned buffers of this rank on the NUMA node its GPU hangs off (the e2e leg moves 1.8 GB per step
    # through them; with 8 ranks on two sockets the remote half would cross the socket link)
    numa_node = L.sj_bind_to_device_numa(local_rank)
    batch = make_batch(args.batch_mib << 20)
    n = len(batch)
    flags = _lib.FLAG_NDJSON | _lib.FLAG_COPY_STRINGS

    # ---- device-resident buffers (torch is only the allocator here) ----
    d_msg = torch.empty(n + (1 << 16), dtype=torch.uint8, device=dev)
    h_in = torch.frombuffer(bytearray(batch), dtype=torch.uint8).pin_memory()
    d_msg[:n].copy_(h_in)
    d_msg[n:] = 0x20
    tcap, scap = C.c_size_t(0), C.c_size_t(0)
    L.sj_bounds(n, C.byref(tcap), C.byref(scap))
    # exact sizes from one functional run through the host API (also the parity anchor of the bench)
    rc, tape_h, strings_h, win = ctx.parse(np.frombuffer(batch, dtype=np.uint8), ndjson=True, copy_strings=True)
    assert rc == 0, rc
    tape_words, string_bytes = len(tape_h), len(strings_h)
    d_tape = torch.empty(tape_words + 64, dtype=torch.int64, device=dev)
    d_strings = torch.empty(string_bytes + 64, dtype=torch.uint8, device=dev)
    tl, sl = C.c_size_t(0), C.c_size_t(0)

    # N > 1: every rank's batch is one shard of ONE NDJSON stream (shards joined by a newline) and the N tapes are the
    # slices of ONE ParsedJson (simdjson_amd64.go:82-93): counting half -> all-gather of the shard totals + exclusive
    # prefix, enqueued on the same stream (no host round trip) -> emitting half with the bases read from device memory
    exchange = "none"
    if world > 1:
        from simdjson_b200.parallel import ShardedParse
        sp = ShardedParse(ctx, device=dev)
        # the exchange as the library's own kernel over peer memory (exchange.cuh): totals pushed into every peer's buffer
        # over NVLink at the end of the counting half, bases left in device memory for the emitting half.  If this box
        # cannot share device memory between processes (CUDA IPC), the same exchange goes through NCCL instead.
        rc_x = sp.connect_exchange(rank, world, gap_bytes=1) if not args.nccl_exchange else -1
        if rc_x == 0:
            exchange = "peer"
            L.sj_exchange_set_timeout_ms(ctx.h, 60000)
        else:
            exchange = "nccl"
            L.sj_ctx_set_stream(ctx.h, torch.cuda.current_stream().cuda_stream)
            my_tot = torch.zeros(4, dtype=torch.int64, device=dev)
            all_tot = torch.zeros(world * 4, dtype=torch.int64, device=dev)
            bases = torch.zeros(3, dtype=torch.int64, device=dev)
            sep = torch.tensor([rank, 0, 0], dtype=torch.int64, device=dev)  # one '\n' between consecutive shards of the message

    def step_device():
        if world == 1:
            r = L.sj_parse_device(ctx.h, d_msg.data_ptr(), n, flags, d_tape.data_ptr(), d_tape.numel(), C.byref(tl),
                                  d_strings.data_ptr(), d_strings.numel(), C.byref(sl))
            assert r == 0, r
            return
        if exchange == "peer":
            r, tot = sp.count(d_msg.data_ptr(), n, True)
            assert r == 0, r
            r = sp.emit(0, 0, 0, d_tape.data_ptr(), d_tape.numel(), d_strings.data_ptr(), d_strings.numel(), sp.bases_ptr)
            assert r == 0, r
            tl.value, sl.value = tot[1], tot[2]
            return
        r, tot = sp.count(d_msg.data_ptr(), n, True, my_tot.data_ptr())
        assert r == 0, r
        dist.all_gather_into_tensor(all_tot, my_tot)          # 4 integers per rank: the path's only exchange
        torch.sum(all_tot.view(world, 4)[:rank, :3], dim=0, out=bases)
        bases.add_(sep)
        r = sp.emit(0, 0, 0, d_tape.data_ptr(), d_tape.numel(), d_strings.data_ptr(), d_strings.numel(), bases.data_ptr())
        assert r == 0, r
        tl.value, sl.value = tot[1], tot[2]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- value: device resident ----
    barrier()  # (the ranks leave their set-up seconds apart; the sharded step is a collective call with a time limit)
    for _ in range(args.warmup):
        step_device()
    ms = C.c_float(0)
    launches0 = ctx.launches()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    L.sj_event_record(ctx.h, 0)
    for _ in range(args.steps):
        step_device()
    L.sj_event_record(ctx.h, 1)
    L.sj_event_elapsed_ms(ctx.h, C.byref(ms))
    barrier()
    launches = ctx.launches() - launches0
    t_dev = reduce_max(ms.value / 1e3)
    assert tl.value == tape_words and sl.value == string_bytes
    if world > 1:
        # the slice is rebased: its first word is this shard's first root, chained to the next one in WHOLE-tape indices
        b_host = sp.exchange_result()[1][:3] if exchange == "peer" else [int(x) for x in bases.tolist()]
        first = int(d_tape[0].item()) & ((1 << 56) - 1)
        assert b_host[1] == rank * tape_words and first == b_host[1] + (int(tape_h[0]) & ((1 << 56) - 1)), (b_host, first)
        if exchange == "nccl":
            L.sj_ctx_set_stream(ctx.h, None)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "_rank%d" % rank if world > 1 else "", DUMP_SAMPLES // world,
                     d_tape, tape_words, d_strings, string_bytes)

    # ---- roofline: stage1_flatten alone on the same batch ----
    info = sj.Stage1Info()
    idx_cap = n // 3 + 1024
    d_idx = torch.empty(idx_cap, dtype=torch.int32, device=dev)
    r = L.sj_stage1_device(ctx.h, d_msg.data_ptr(), n, 1, 0, d_idx.data_ptr(), idx_cap, C.byref(info))
    assert r == 0 and not info.overflow
    for _ in range(3):
        L.sj_stage1_launch(ctx.h, d_msg.data_ptr(), n, 1, 0, d_idx.data_ptr(), idx_cap)
    L.sj_ctx_sync(ctx.h)
    L.sj_event_record(ctx.h, 0)
    for _ in range(args.steps):
        L.sj_stage1_launch(ctx.h, d_msg.data_ptr(), n, 1, 0, d_idx.data_ptr(), idx_cap)
    L.sj_event_record(ctx.h, 1)
    L.sj_event_elapsed_ms(ctx.h, C.byref(ms))
    t_s1 = ms.value / 1e3 / args.steps
    alg_bytes = n + 4 * int(info.n_idx)
    peak, peak_kind = read_peaks()
    achieved = alg_bytes / t_s1 / 1e9

    # ---- roofline_twitter: the input the north-star target is stated on (SURVEY.md 8d, S1): "[" + twitter.json x K + "]",
    # >= 1 GiB (> L2), one valid document, K1 alone.  Rank 0 at N = 1 only (the other N re-use the N = 1 figure).
    roof_tw = None
    if world == 1 and args.twitter_mib > 0:
        from tests.util import load_fixture
        tw = load_fixture("twitter").strip()
        k = max(1, (args.twitter_mib << 20) // (len(tw) + 1))
        doc = b"[" + b",".join([tw] * k) + b"]"
        n_tw = len(doc)
        d_tw = torch.empty(n_tw + (1 << 16), dtype=torch.uint8, device=dev)
        d_tw[:n_tw].copy_(torch.frombuffer(bytearray(doc), dtype=torch.uint8))
        d_tw[n_tw:] = 0x20
        del doc
        cap_tw = n_tw // 6 + 1024
        d_idx_tw = torch.empty(cap_tw, dtype=torch.int32, device=dev)
        info_tw = sj.Stage1Info()
        r = L.sj_stage1_device(ctx.h, d_tw.data_ptr(), n_tw, 0, 0, d_idx_tw.data_ptr(), cap_tw, C.byref(info_tw))
        assert r == 0 and not info_tw.overflow and not info_tw.error and int(info_tw.n_idx) == 55263 * k + (k - 1) + 2, (r, info_tw.n_idx)
        for _ in range(3):
            L.sj_stage1_launch(ctx.h, d_tw.data_ptr(), n_tw, 0, 0, d_idx_tw.data_ptr(), cap_tw)
        L.sj_ctx_sync(ctx.h)
        L.sj_event_record(ctx.h, 0)
        for _ in range(args.steps):
            L.sj_stage1_launch(ctx.h, d_tw.data_ptr(), n_tw, 0, 0, d_idx_tw.data_ptr(), cap_tw)
        L.sj_event_record(ctx.h, 1)
        L.sj_event_elapsed_ms(ctx.h, C.byref(ms))
        t_tw = ms.value / 1e3 / args.steps
        alg_tw = n_tw + 4 * int(info_tw.n_idx)
        roof_tw = {"bound": "hbm", "kernel": "stage1_flatten_kernel<single document>", "workload": "twitter.json-shaped: '[' + twitter.json x %d + ']' (SURVEY.md 8d S1), %d bytes, %d structurals (= 55 263 per copy, G8)" % (k, n_tw, int(info_tw.n_idx)),
                   "achieved": round(alg_tw / t_tw / 1e9, 2), "peak": peak, "unit": "GB/s", "frac": round(alg_tw / t_tw / 1e9 / peak, 4),
                   "peak_kind": peak_kind, "algorithmic_bytes_per_launch": alg_tw, "ms_per_launch": round(t_tw * 1e3, 4),
                   "input_read_gbs": round(n_tw / t_tw / 1e9, 2), "input_read_frac": round(n_tw / t_tw / 1e9 / peak, 4),
                   "timer": "CUDA events on the library's stream around %d back-to-back launches" % args.steps}
        del d_tw, d_idx_tw
        torch.cuda.empty_cache()

    # ---- e2e: host buffers through sj_parse (pinned in, pinned out) ----
    # ParseNDStream keeps several chunks in flight (simdjson_amd64.go:132); here `--inflight`
    # host threads each own a context (= CUDA stream) and their own pinned output buffers, so
    # the H2D copy, the kernels and the D2H copy of consecutive batches overlap.
    workers = []
    for w in range(max(1, args.inflight)):
        wctx = ctx if w == 0 else sj.Context(local_rank)
        workers.append({"ctx": wctx, "tape": torch.empty(tape_words + 64, dtype=torch.int64).pin_memory(),
                        "strings": torch.empty(string_bytes + 64, dtype=torch.uint8).pin_memory()})

    def step_host(w, fl=flags, want_strings=None):
        tl2, sl2, mo, ml = C.c_size_t(0), C.c_size_t(0), C.c_size_t(0), C.c_size_t(0)
        r = L.sj_parse(w["ctx"].h, h_in.data_ptr(), n, fl, w["tape"].data_ptr(), w["tape"].numel(), C.byref(tl2),
                       w["strings"].data_ptr(), w["strings"].numel(), C.byref(sl2), C.byref(mo), C.byref(ml))
        assert r == 0 and tl2.value == tape_words, r
        if want_strings is not None:
            assert sl2.value == want_strings, sl2.value

    def run_host_steps(count, fl=flags, want_strings=None):
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=len(workers)) as ex:
            futs = [ex.submit(lambda k=k: [step_host(workers[k], fl, want_strings) for _ in range(k, count, len(workers))])
                    for k in range(len(workers))]
            for f in futs:
                f.result()

    run_host_steps(max(args.warmup, len(workers)))
    barrier()
    t0 = time.perf_counter()
    run_host_steps(args.steps)
    torch.cuda.synchronize()
    t_e2e = reduce_max(time.perf_counter() - t0)
    barrier()
    for w in workers[: min(len(workers), args.steps)]:
        assert np.array_equal(w["tape"][:tape_words].numpy().view(np.uint64), tape_h)

    # the same call with WithCopyStrings(false) (options.go:13): strings stay in the message unless they hold escapes, so
    # only the tape travels back (this stream has no escapes: Strings.B is empty)
    fl_nc = _lib.FLAG_NDJSON
    rc_nc, tape_nc, strings_nc, _ = ctx.parse(np.frombuffer(batch, dtype=np.uint8), ndjson=True, copy_strings=False)
    assert rc_nc == 0 and len(tape_nc) == tape_words
    run_host_steps(max(args.warmup, len(workers)), fl_nc, len(strings_nc))
    barrier()
    t0 = time.perf_counter()
    run_host_steps(args.steps, fl_nc, len(strings_nc))
    torch.cuda.synchronize()
    t_e2e_nc = reduce_max(time.perf_counter() - t0)
    barrier()

    # ---- stream: BASELINE configs[4] as the reference runs it -- ParseNDStream (simdjson_amd64.go:116-215) -- through the
    # LIBRARY's own pipeline (sj_stream_*: chunks cut at record boundaries, pinned staging, one context + worker per
    # slot, ordered delivery), not through Python threads.  The records come from K0 (gen_ndjson): record g = template
    # line g mod 1000 with Ticket := g, so every record of this rank's ring is different; `--stream-gib` GiB per GPU-set
    # (64) are pushed by cycling over the ring. ----
    stream_line = None
    if args.stream_gib > 0:
        tmpl = load_records() + b"\n"
        ring_cap = args.stream_ring_mib << 20
        n_rec = max(1000, (ring_cap // len(tmpl)) * 1000)
        d_ring = torch.empty(ring_cap + (4 << 20), dtype=torch.uint8, device=dev)
        glen = C.c_size_t(0)
        r = L.sj_gen_ndjson_device(ctx.h, tmpl, len(tmpl), rank * n_rec, n_rec, d_ring.data_ptr(), d_ring.numel(), C.byref(glen))
        assert r == 0, r
        ring_len = glen.value + 1
        d_ring[glen.value] = 0x0A  # the ring ends with a newline, so it can be pushed round and round
        h_ring = torch.empty(ring_len, dtype=torch.uint8).pin_memory()
        h_ring.copy_(d_ring[:ring_len])
        torch.cuda.synchronize()
        first = bytes(h_ring[:40].numpy().tobytes())
        assert first.startswith(b'{"Ticket":"%010d"' % ((rank * n_rec) % 10**10)), first
        del d_ring
        torch.cuda.empty_cache()
        total_push = (args.stream_gib << 30) // world
        hs = C.c_void_p()
        r = L.sj_stream_create(local_rank, max(2, args.inflight), args.stream_chunk_mib << 20, _lib.FLAG_COPY_STRINGS, C.byref(hs))
        assert r == 0, r
        res = _lib.StreamResult()
        taken = C.c_size_t(0)
        st = {"chunks": 0, "msg": 0, "tape": 0, "strings": 0}

        def take_one():
            rr = L.sj_stream_next(hs, C.byref(res))
            if rr == 0:
                st["chunks"] += 1
                st["msg"] += res.message_len
                st["tape"] += res.tape_len
                st["strings"] += res.strings_len
                L.sj_stream_release(hs, C.byref(res))
            return rr

        def push(nbytes):
            pos, left = push.pos, nbytes
            while left > 0:
                n1 = min(left, ring_len - pos, 64 << 20)
                rr = L.sj_stream_write(hs, h_ring.data_ptr() + pos, n1, C.byref(taken))
                assert rr == 0, rr
                pos = (pos + taken.value) % ring_len
                left -= taken.value
                if taken.value == 0:
                    assert take_one() == 0
            push.pos = pos

        push.pos = 0
        push(min(total_push, 2 * (args.stream_chunk_mib << 20)))  # warm the slots' buffers up
        barrier()
        t0 = time.perf_counter()
        push(total_push)
        while True:
            rr = L.sj_stream_close_input(hs)
            if rr != _lib.STREAM_BUSY:
                break
            assert take_one() == 0
        assert rr == 0, rr
        while take_one() == 0:
            pass
        t_stream = reduce_max(time.perf_counter() - t0)
        barrier()
        L.sj_stream_destroy(hs)
        pushed = total_push + min(total_push, 2 * (args.stream_chunk_mib << 20))
        assert abs(st["msg"] - pushed) <= 2 * st["chunks"] + ring_len, (st, pushed)  # everything pushed came back parsed (minus trimmed newlines / the tail)
        stream_line = {"value": round(total_push * world / t_stream / 1e9, 3), "unit": "GB/s", "bytes_per_gpu": total_push,
                       "seconds": round(t_stream, 3), "chunks_per_gpu": st["chunks"], "chunk_mib": args.stream_chunk_mib,
                       "slots": max(2, args.inflight), "ring_mib": ring_len >> 20, "records_in_ring": n_rec,
                       "tape_words_per_gpu": st["tape"], "string_bytes_per_gpu": st["strings"],
                       "what": "sj_stream_* (the library's ParseNDStream): host bytes pushed with sj_stream_write, results taken in order "
                               "from pinned slot buffers with sj_stream_next; unique records from K0 gen_ndjson; host wall clock, max over ranks"}
        del h_ring

    # ---- tape consumer on the device (SURVEY.md 8f): parseMessage + countWhere("Make", "HOND"), the reference's
    # BenchmarkNdjsonColdCountStarWithWhere (parse_json_amd64_test.go:134): host input, only two counts come back ----
    n_records = batch.count(b"\n") + 1
    cw_seen = []

    def step_count(w):
        roots, matches = C.c_uint64(0), C.c_uint64(0)
        r = L.sj_parse_count_where(w["ctx"].h, h_in.data_ptr(), n, flags, b"Make", 4, b"HOND", 4, C.byref(roots), C.byref(matches))
        assert r == 0 and roots.value == n_records, (r, roots.value)
        cw_seen.append(matches.value)

    def run_count_steps(count):
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=len(workers)) as ex:
            futs = [ex.submit(lambda k=k: [step_count(workers[k]) for _ in range(k, count, len(workers))])
                    for k in range(len(workers))]
            for f in futs:
                f.result()

    run_count_steps(max(args.warmup, len(workers)))
    barrier()
    t0 = time.perf_counter()
    run_count_steps(args.steps)
    torch.cuda.synchronize()
    t_cw = reduce_max(time.perf_counter() - t0)
    barrier()
    assert len(set(cw_seen)) == 1 and cw_seen[0] == 116 * (n_records // 1000), cw_seen[:3]  # ndjson_test.go:263 per 1000 records
    sampler.stop_flag = True
    sampler.join(timeout=3)

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of the same stream ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads, quota = host_threads()
        sample = batch
        while len(sample) < (args.cpu_sample_mib << 20):
            sample = sample + b"\n" + batch
        sample = sample[: args.cpu_sample_mib << 20]
        sample = sample[: sample.rfind(b"\n")]
        warm = sample[: 32 << 20]
        cpu_parse_stream(warm[: warm.rfind(b"\n")], threads)
        cpu_parse_stream(sample, threads)  # first touch of every worker's buffers stays outside the timed region
        secs, nb = cpu_parse_stream(sample, threads)
        reps = 1
        while secs < 5.0 and reps < 8:  # stretch tiny timings to a few seconds of CPU work
            t2, n2 = cpu_parse_stream(sample, threads)
            secs += t2
            nb += n2
            reps += 1
        t_c, n_c = cpu_parse_stream(sample, threads, count_where=(b"Make", b"HOND"))
        cpu = {"value": round(nb / secs / 1e9, 4), "unit": "GB/s", "cores": threads, "kind": "port", "isa": _cpu_isa,
               "sample": "%d x %d MiB of the same NDJSON stream, 10 MiB chunks on all host threads (oracle port, %s mask routines; the Go reference cannot be built here) %s" % (reps, len(sample) >> 20, _cpu_isa, quota),
               "parse_count_where": round(n_c / t_c / 1e9, 4)}

    if rank == 0:
        total_bytes = n * world * args.steps
        line = {
            "metric": METRIC,
            "value": round(total_bytes / t_dev / 1e9, 3), "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(t_dev / args.steps * 1e3, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "batch_bytes_per_gpu": n, "records_per_batch": batch.count(b"\n") + 1, "tape_words": tape_words,
                       "string_bytes": string_bytes, "inputs_larger_than_l2": True, "parallelism": "ndjson-shard x%d" % world,
                       "collective": {"none": "none",
                                      "peer": "the library's own exchange kernel (exchange.cuh): each rank's counting half ends with one warp that stores the shard totals (4 x u64) into every peer's buffer over NVLink (CUDA IPC peer memory), polls its local buffer for the peers' and leaves the bases of ONE ParsedJson in device memory for the emitting half; no NCCL on the data path",
                                      "nccl": "all_gather of 4 x int64 per rank per step (shard totals -> bases of ONE ParsedJson), enqueued on the parse's stream between sj_parse_nd_sharded_count and _emit"}[exchange],
                       "numa_node_bound": int(numa_node)},
            "e2e": {"value": round(total_bytes / t_e2e / 1e9, 3), "unit": "GB/s", "h2d_bytes_per_step": n,
                    "d2h_bytes_per_step": tape_words * 8 + string_bytes, "ms_per_step": round(t_e2e / args.steps * 1e3, 3),
                    "calls_in_flight": len(workers), "timer": "host wall clock around the in-flight calls, device synchronised on both sides"},
            "e2e_nocopy": {"value": round(total_bytes / t_e2e_nc / 1e9, 3), "unit": "GB/s", "h2d_bytes_per_step": n,
                           "d2h_bytes_per_step": tape_words * 8 + len(strings_nc), "ms_per_step": round(t_e2e_nc / args.steps * 1e3, 3),
                           "what": "the same sj_parse calls with WithCopyStrings(false) (options.go:13): the tape alone travels back"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "stage1_flatten_kernel<ndjson>", "achieved": round(achieved, 2), "peak": peak,
                         "unit": "GB/s", "frac": round(achieved / peak, 4), "peak_kind": peak_kind, "traffic": k1_traffic(n),
                         "traffic_kind": "static: dram__bytes_read.sum + dram__bytes_write.sum of one K1 launch on this batch from the committed ncu --set full capture (profiles/k1_traffic.json, round 2), not measured in this run",
                         "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": round(t_s1 * 1e3, 4),
                         "input_read_gbs": round(n / t_s1 / 1e9, 2)},
            "roofline_parse": {"bound": "hbm", "what": "whole device-resident step (K1 + K2p/q/r + numbers, scope matching, links, roots), algorithmic bytes 2*N_in + 8*N_idx + 8*N_tape + N_strings (SURVEY.md 8d)",
                               "achieved": round((2 * n + 8 * int(info.n_idx) + 8 * tape_words + string_bytes) * world * args.steps / t_dev / 1e9, 2),
                               "peak": peak, "unit": "GB/s",
                               "frac": round((2 * n + 8 * int(info.n_idx) + 8 * tape_words + string_bytes) * args.steps / t_dev / 1e9 / peak, 4)},
            "parse_count_where": {"value": round(total_bytes / t_cw / 1e9, 3), "unit": "GB/s", "ms_per_step": round(t_cw / args.steps * 1e3, 3),
                                  "h2d_bytes_per_step": n, "d2h_bytes_per_step": 16, "records": n_records, "matches": int(cw_seen[0]),
                                  "what": "sj_parse_count_where: host NDJSON in, parse + countWhere(Make == HOND) on the device "
                                          "(parse_json_amd64_test.go:134), tape stays in HBM; same in-flight scheme and timer as e2e"},
            "clocks": sampler.summary(),
        }
        if roof_tw:
            line["roofline_twitter"] = roof_tw
        if stream_line:
            line["stream"] = stream_line
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
