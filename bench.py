#!/usr/bin/env python
"""Headline benchmark: .et encode + decode throughput (uncompressed GB/s) against the HBM roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

A step = one encode (histogram -> host codebook -> pack) followed by one decode (dictionary parse
-> self-synchronising decode) of the workload, both through the C ABI (include/entreepy_b200.h).
`value` = uncompressed bytes per step / device time per step with the input resident in HBM;
`e2e` = the same through et_encode/et_decode with pinned HOST buffers (H2D and D2H inside the
timed region).  Workloads are BASELINE.md §4's (synthetic, splitmix64 seed 0xE7C0DE):
    N=1 default  text-1G  (2^30 B, the config the per-B200 roofline is quoted on)
    N>1 default  text-4G  (2^32-16 B, one .et stream sharded over the ranks: strong scaling)
Inputs are far larger than the 126 MB L2, so no explicit flush between iterations.

--impl reference times the reference ALGORITHM on the host (oracle/entreepy_oracle.c, a C
restatement: the reference is Zig and no Zig toolchain exists here or on the GPU box — there is no
oracle/_ref), single thread like the reference, on a bounded sample of the same workload.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "encode+decode round-trip GB/s (uncompressed)"
WORKLOADS = {  # name -> (bytes, weights kind)
    "midsummer": (112541, "file"),
    "text-5M": (5452595, "text"),
    "text-256M": (1 << 28, "text"),
    "text-1G": (1 << 30, "text"),
    "text-4G": ((1 << 32) - 16, "text"),
    "uniform256": (1 << 28, "uniform256"),
    "uniform255": (1 << 28, "uniform255"),
    "fib32": (1 << 28, "fib32"),
}
CPU_SAMPLE = 96 << 20       # bytes of the workload the cpu_baseline leg runs (about 10 s of host work)
REF_SAMPLE = 32 << 20       # bytes per step of the --impl reference arm (about 2.5 s per step)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def manifest():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "manifest.json")))


def thresholds(kind):
    from entreepy_b200 import synth

    if kind == "text":
        w = synth.text_weights(manifest()["midsummer_histogram"])
    elif kind == "uniform256":
        w = synth.uniform_weights(0)
    elif kind == "uniform255":
        w = synth.uniform_weights(1)
    elif kind == "fib32":
        w = synth.fibonacci_weights(32)
    else:
        raise ValueError(kind)
    return synth.thresholds_from_weights(w)


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_for(kernels, workload="text-1G"):
    """dram bytes (read + write) of one launch of each of `kernels`, summed, from the committed ncu --set full
    capture of this workload (profiles/traffic.json, written by tools/profile_summary.py); None if not captured."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(workload, {})
        vals = [t[k] for k in kernels]
        return int(sum(vals))
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8:
                self.rows.append(f)

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
            self.t.join(timeout=2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[4 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ---------------------------------------------------------------------------------- host baseline
def host_sample(kind, n):
    from entreepy_b200 import synth

    if kind == "file":
        return np.frombuffer(open(os.path.join(ROOT, "tests", "golden", "a_midsummer_nights_dream.txt"), "rb").read(),
                             dtype=np.uint8)[:n]
    return synth.generate(n, thresholds(kind))


def time_oracle(sample):
    """One encode + one decode of `sample` with the C restatement of the reference algorithm."""
    from oracle import oracle

    t0 = time.perf_counter()
    enc = oracle.encode(sample, cap=9000 + 5 * sample.size)
    t1 = time.perf_counter()
    rc, dec = oracle.decode_ref(enc[4:], sample.size)  # decode.zig's algorithm (hash probe per length)
    which = "decode.zig restatement"
    if rc != 0 or dec.size != sample.size:
        # the reference decoder cannot decode this stream (SURVEY §0.5): time the plain trie decoder instead
        t1 = time.perf_counter()
        dec = oracle.decode(enc[4:], sample.size)
        which = "bit-serial trie decoder (reference decoder fails on this input)"
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, which


def run_reference(args, rank):
    if rank != 0:
        return 0
    n_total, kind = WORKLOADS[args.workload]
    n = min(n_total, REF_SAMPLE)
    sample = host_sample(kind, n)
    times = []
    which = ""
    for i in range(args.warmup + args.steps):
        te, td, which = time_oracle(sample)
        if i >= args.warmup:
            times.append((te, td))
    te = sum(t[0] for t in times) / len(times)
    td = sum(t[1] for t in times) / len(times)
    value = n / 1e9 / (te + td)
    sample_desc = f"first {n} B of {args.workload}, encode + decode per step; decode = {which}"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": (te + td) * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": args.workload, "bytes": n_total, "sample_bytes": n},
        "encode_gbs": n / 1e9 / te, "decode_gbs": n / 1e9 / td,
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": 1, "kind": "port", "sample": sample_desc,
                         "note": "C restatement of the reference algorithm (oracle/entreepy_oracle.c); the reference is "
                                 "Zig and cannot be built here (no Zig toolchain); its compute is single-threaded"},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------- GPU arm
class OneGpu:
    """N=1: the drop-in entry points et_encode_dev / et_decode_dev on one whole stream."""

    def __init__(self, codec, n, stream):
        import torch

        from entreepy_b200 import _abi

        self.codec, self.n, self.stream = codec, n, stream
        self.enc = torch.empty(n + 16384, dtype=torch.uint8, device="cuda")
        self.dec = torch.empty(n + 16, dtype=torch.uint8, device="cuda")
        self.flags = _abi.FLAG_WRITE_OUTPUT | _abi.FLAG_TIMING
        self.size = 0

    def encode(self, inp):
        self.size = self.codec.encode_dev(inp.data_ptr(), self.n, self.enc.data_ptr(), self.enc.numel(), self.flags, self.stream)
        return self.size - self.header_bytes()

    def header_bytes(self):
        if not hasattr(self, "_hb"):
            import entreepy_b200 as et

            self._hb = 4 + int(et.parse_header(self.enc[4:4100].cpu().numpy()).body_offset)
        return self._hb

    def prepare_decode(self):
        pass

    def decode(self):
        got = self.codec.decode_dev(self.enc.data_ptr() + 4, self.size - 4, self.dec.data_ptr(), self.n, self.flags, self.stream)
        return got, 0

    def outputs(self, got, offset):
        """What the callers of et_encode_dev / et_decode_dev received in the last step."""
        return {"encoded": self.enc[: self.size], "decoded": self.dec[:got]}, [self.size, got]

    def e2e_buffers(self):
        c = self.codec
        return c.pinned(self.n), c.pinned(self.n + 16384), c.pinned(self.n)

    def e2e_step(self, h_in, h_enc, h_dec):
        import entreepy_b200 as et

        size = self.codec.encode_into(h_in, h_enc, et.EncodeFlags(write_output=True))
        got = self.codec.decode_into(h_enc[4:size], h_dec, et.DecodeFlags(write_output=True))
        return got, int(self.n + size - 4), int(size + self.n)


class ManyGpus:
    """N>1: one stream sharded over the ranks (entreepy_b200.sharded on the shard entry points)."""

    def __init__(self, codec, plan, dist, stream, py_exchange=False):
        import torch

        from entreepy_b200 import sharded

        self.codec, self.plan, self.dist = codec, plan, dist
        py_comm = sharded.Comm(dist, torch.device("cuda"))
        if py_exchange:  # the exchanges in Python over torch.distributed (round 1's path, kept for comparison)
            self.coder = sharded.ShardedCodec(sharded.GpuBackend(codec, stream), plan, py_comm)
            self.path = "entreepy_b200.sharded.ShardedCodec (exchanges in Python over torch.distributed)"
        else:  # the whole protocol behind the C ABI, its all-gathers on an NCCL communicator of the library's own
            uid = [codec.comm_unique_id() if plan.rank == 0 else None]
            dist.broadcast_object_list(uid, 0)
            self.ncomm = codec.comm_nccl(uid[0], plan.rank, plan.world)
            self.coder = sharded.NativeShardedCodec(codec, plan, self.ncomm, py_comm, stream)
            self.path = "et_encode_sharded_dev + et_decode_sharded_dev (C ABI, ncclAllGather on the context's stream)"
        self.body = torch.empty(plan.n_local + 16384, dtype=torch.uint8, device="cuda")
        self.res = self.range = self.dec = None

    def encode(self, inp):
        self.res = self.coder.encode(inp, self.body)
        return self.res.own_hi - self.res.own_lo

    def prepare_decode(self):
        """What a file reader would do: give every rank its equal share of the body (untimed setup)."""
        import torch

        self.range = self.coder.scatter_body(self.res, self.body).clone()
        cuts, ranges = self.coder.decode_ranges(self.res.body_bytes)
        self.own_body = cuts[self.plan.rank + 1] - cuts[self.plan.rank]
        # text of an equal share of the body: about n_total / world symbols; leave generous room
        self.dec = torch.empty(int(self.plan.n_total / self.plan.world * 1.25) + (1 << 20), dtype=torch.uint8, device="cuda")

    def decode(self):
        d = self.coder.decode(self.res.header[4:], self.res.body_bytes, self.range, self.dec)
        self.rounds = d.rounds
        return d.n_local, d.offset

    def outputs(self, got, offset):
        """What this rank's caller received in the last step: the .et header, the body bytes [own_lo, own_hi) it
        holds, and the text it decoded, which starts at `offset` of the original."""
        import torch

        res = self.res
        header = torch.frombuffer(bytearray(res.header), dtype=torch.uint8)
        body = self.body[res.own_lo - res.first_byte : res.own_hi - res.first_byte]
        return {"header": header, "encoded": body, "decoded": self.dec[:got]}, [res.own_lo, res.own_hi, offset, got]

    def e2e_buffers(self):
        import torch

        return (torch.empty(self.plan.n_local, dtype=torch.uint8).pin_memory(),
                torch.empty(self.body.numel(), dtype=torch.uint8).pin_memory(),
                (torch.empty(self.range.numel(), dtype=torch.uint8).pin_memory(),
                 torch.empty(self.dec.numel(), dtype=torch.uint8).pin_memory()))

    def e2e_step(self, h_in, h_body, h_pair, inp):
        import torch

        h_range, h_text = h_pair
        if not hasattr(self, "_side"):
            self._side = torch.cuda.Stream()
        inp[: self.plan.n_local].copy_(h_in, non_blocking=True)
        res = self.coder.encode(inp, self.body)  # returns with the stream idle
        nb = res.own_hi - res.own_lo
        # the link is full duplex: the body goes down on a second stream while the decoder's input comes up
        with torch.cuda.stream(self._side):
            h_body[:nb].copy_(self.body[res.own_lo - res.first_byte : res.own_hi - res.first_byte], non_blocking=True)
        self.range.copy_(h_range, non_blocking=True)
        d = self.coder.decode(res.header[4:], res.body_bytes, self.range, self.dec)
        h_text[: d.n_local].copy_(self.dec[: d.n_local], non_blocking=True)
        torch.cuda.synchronize()
        return d.n_local, int(self.plan.n_local + self.range.numel()), int(nb + d.n_local)


def bind_to_gpu_numa_node(index):
    """Pins this rank to the CPUs NVML reports as local to its GPU, so that its page-locked staging buffers are
    allocated on that socket: with 8 ranks copying at once the host's memory controllers and the inter-socket link are
    what the end-to-end number hits first.  Returns a short description (None when the affinity cannot be read/set)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {i for i in range(os.cpu_count()) if (mask[i // 64] >> (i % 64)) & 1}
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return f"{len(allowed)} cpus local to gpu {index}"
    except Exception:
        return None


def verify_one(codec, arm, inp, n, got, kind):
    """decode(encode(x)) == x on one GPU (north_star)."""
    import torch

    import entreepy_b200 as et

    verified = got == n and bool(torch.equal(arm.dec[:n], inp[:n]))
    if not verified and kind == "uniform256":
        # all 256 byte values occur: the reference encoder gives the last symbol in sort order no code
        # (encode.zig:70, SURVEY §0.2), so the round trip is the text WITHOUT that symbol — by construction
        counts = codec.histogram_dev(inp.data_ptr(), n)
        cb = et.build_codebook(counts)
        dropped = [s for s in range(256) if counts[s] and cb.code[s].length == 0]
        keep = inp[:n][inp[:n] != dropped[0]] if len(dropped) == 1 else inp[:0]
        verified = len(dropped) == 1 and got == keep.numel() and bool(torch.equal(arm.dec[:got], keep))
    return verified


def make_input(codec, name, lo=0, n=None, world=1):
    """The workload's bytes [lo, lo + n) on the device (same bytes as entreepy_b200/synth.py on the CPU)."""
    import torch

    from entreepy_b200 import synth

    n_total, kind = WORKLOADS[name]
    n = n_total if n is None else n
    inp = torch.empty(n + 16, dtype=torch.uint8, device="cuda")
    if kind == "file":
        inp[:n].copy_(torch.from_numpy(host_sample(kind, n_total)[lo:lo + n].copy()))
    elif kind == "fib32" and world == 1:
        # exact counts, shuffled (SURVEY §0.4): the Huffman tree is a chain of depth 32 — i.i.d. sampling is not
        inp[:n].copy_(synth.shuffled_dev(synth.fibonacci_counts(n, 32)))
    else:
        codec.synth_dev(inp.data_ptr(), n, synth.SEED, lo, thresholds(kind))
    torch.cuda.synchronize()
    return inp


OTHER_CONFIGS = ["midsummer", "text-5M", "uniform255", "uniform256", "fib32", "text-4G"]  # BASELINE.json configs 1, 2, 4, 5


def run_other_configs(codec, stream, peak, steps=3):
    """BASELINE.json's other configurations on one GPU, device resident, outside the headline's timed region:
    encode and decode milliseconds (CUDA events, mean of `steps` after two warm-up steps), fraction of the HBM
    roofline in algorithmic bytes (2N + C, C + N), fixpoint rounds of the decoder, round trip checked."""
    import torch

    out = []
    for name in OTHER_CONFIGS:
        n, kind = WORKLOADS[name]
        try:
            inp = make_input(codec, name)
            arm = OneGpu(codec, n, stream)
            enc_ms, dec_ms, got, c = [], [], 0, 0
            for i in range(2 + steps):
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                e0.record()
                c = arm.encode(inp)
                e1.record()
                got, _ = arm.decode()
                e2.record()
                torch.cuda.synchronize()
                if i >= 2:
                    enc_ms.append(e0.elapsed_time(e1))
                    dec_ms.append(e1.elapsed_time(e2))
            te, td = statistics.mean(enc_ms), statistics.mean(dec_ms)
            row = {"workload": name, "bytes": n, "compressed_bytes": int(c), "encode_ms": te, "decode_ms": td,
                   "encode_gbs": n / 1e6 / te, "decode_gbs": n / 1e6 / td, "round_trip_gbs": n / 1e6 / (te + td),
                   "encode_frac": (2 * n + c) / 1e6 / te / peak, "decode_frac": (c + got) / 1e6 / td / peak,
                   "rounds": codec.last_decode_rounds, "verified_round_trip": verify_one(codec, arm, inp, n, got, kind)}
            if n < (126 << 20):
                row["note"] = "fits the 126 MB L2: launch-latency bound, the HBM fraction is not meaningful"
            if kind == "uniform256":
                row["note"] = "all 256 byte values: the reference drops one symbol (encode.zig:70); round trip == text without it"
            out.append(row)
            del arm, inp
            torch.cuda.empty_cache()
        except Exception as exc:  # a config that cannot run must not take the headline down with it
            out.append({"workload": name, "error": f"{type(exc).__name__}: {exc}"})
    return out


DUMP_VALUES = 12 << 20  # float32 values --dump-outputs writes, all ranks together (48 MB of the 64 MB it may write)
DUMP_BLOCK = 1 << 20    # bytes per block sum of an output written as a sample


def dump_outputs(path, outputs, sizes, rank, world):
    """--dump-outputs: the byte arrays the timed path returned in its last step, as .npy files, so that two builds
    can be compared output for output.  <name>.npy holds the bytes as float32: the whole array when it is short,
    otherwise the bytes at positions numpy.random.default_rng(0).integers(0, len, k), sorted, plus <name>_block_sums.npy
    (float64), the sum of every DUMP_BLOCK bytes, so that a change anywhere shows.  sizes.npy (float64) holds the
    counts the calls returned.  With N > 1 every rank writes its own files, suffixed _rank<r>."""
    import torch

    os.makedirs(path, exist_ok=True)
    tag = f"_rank{rank}" if world > 1 else ""
    k = DUMP_VALUES // (len(outputs) * world)
    for name, t in outputs.items():
        n = t.numel()
        vals = t
        if n > k:
            idx = np.sort(np.random.default_rng(0).integers(0, n, k))
            vals = t[torch.from_numpy(idx).to(t.device)]
            whole = n // DUMP_BLOCK * DUMP_BLOCK
            sums = [t[:whole].view(-1, DUMP_BLOCK).sum(dim=1, dtype=torch.int64).cpu()]
            if whole < n:
                sums.append(t[whole:].sum(dtype=torch.int64).view(1).cpu())
            np.save(os.path.join(path, f"{name}_block_sums{tag}.npy"), torch.cat(sums).numpy().astype(np.float64))
        np.save(os.path.join(path, f"{name}{tag}.npy"), vals.float().cpu().numpy())
    np.save(os.path.join(path, f"sizes{tag}.npy"), np.array(sizes, dtype=np.float64))


def run_ours(args, rank, world):
    import torch

    import entreepy_b200 as et
    from entreepy_b200 import sharded, synth

    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference for the host baseline)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None  # before any pinned allocation: first touch decides the node
    dist = None
    if world > 1:
        import torch.distributed as dist

        # the communicator prints "NCCL version ..." on stdout when it is created: stdout carries one JSON line only
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    codec = et.Codec(local)
    if os.environ.get("ET_BENCH_DEBUG"):  # developer switch: ET_TUNE_DEBUG bits (per-phase timing lines on stderr)
        codec.set_tuning(et._abi.TUNE_DEBUG, int(os.environ["ET_BENCH_DEBUG"]))
    n_total, kind = WORKLOADS[args.workload]
    plan = sharded.ShardPlan(n_total, world, rank)
    n = plan.n_local
    stream = torch.cuda.current_stream().cuda_stream
    thr = thresholds(kind) if kind != "file" else None
    inp = make_input(codec, args.workload, plan.lo, n, world)
    arm = OneGpu(codec, n, stream) if world == 1 else ManyGpus(codec, plan, dist, stream, args.py_exchange)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step(stats=None, events=None):
        # (the timed loop hands in events made beforehand: creating three per step costs more host time than the
        # step's own launches at 8 GPUs)
        e0, e1, e2 = events if events is not None else (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        c_local = arm.encode(inp)
        ms_enc = codec.last_stage_ms()
        if world > 1:  # the shard call times only its pack; the histogram is a call of its own
            ms_enc[0] = getattr(arm.coder.backend, "hist_ms", 0.0)
        e1.record()
        got, offset = arm.decode()
        ms_dec = codec.last_stage_ms() + [codec.last_decode_rounds]
        e2.record()
        if stats is not None:
            stats.append((e0, e1, e2, ms_enc, ms_dec))
        return c_local, got, offset

    c_local = arm.encode(inp)
    arm.prepare_decode()
    for _ in range(max(args.warmup, 3)):
        c_local, got, offset = step()
    barrier()
    # round trip == original (north_star): the text this rank decoded is text[offset : offset + got]
    if world == 1:
        verified = verify_one(codec, arm, inp, n, got, kind)
    else:
        want = torch.empty(got + 16, dtype=torch.uint8, device="cuda")
        if kind == "file":
            want[:got].copy_(torch.from_numpy(host_sample(kind, n_total)[offset:offset + got].copy()))
        else:
            codec.synth_dev(want.data_ptr(), got, synth.SEED, offset, thr)
        ok = torch.tensor([int(torch.equal(arm.dec[:got], want[:got])), got], dtype=torch.int64, device="cuda")
        dist.all_reduce(ok)
        verified = int(ok[0].item()) == world and int(ok[1].item()) == n_total
        del want
    if not verified:
        raise SystemExit("bench.py: decode(encode(x)) != x — refusing to report a throughput")

    stats = []
    with ClockSampler(local) as clocks:
        # nvidia-smi takes a few hundred ms to deliver its first row and the timed region may be shorter than that
        # (8 GPUs: ~2 ms per step): keep the same load running, untimed, until samples arrive, so that the clocks
        # line describes the GPU under this load
        t_wait = time.perf_counter()
        while True:
            done = len(clocks.rows) >= 3 or time.perf_counter() - t_wait >= 3.0 or clocks.proc is None
            if dist is not None:  # rank 0 decides: every rank takes the same number of steps
                flag = torch.tensor([int(done)], device="cuda")
                dist.broadcast(flag, 0)
                done = bool(int(flag.item()))
            if done:
                break
            step()
        launches0 = codec.kernel_launches
        step_events = [tuple(torch.cuda.Event(enable_timing=True) for _ in range(3)) for _ in range(args.steps)]
        for ev in step_events:  # (an event is created by its first record)
            for e in ev:
                e.record()
        barrier()
        t_begin = torch.cuda.Event(enable_timing=True)
        t_end = torch.cuda.Event(enable_timing=True)
        t_begin.record()
        for ev in step_events:
            c_local, got, offset = step(stats, ev)
        t_end.record()
        barrier()
    if args.dump_outputs:  # before the end-to-end leg, which reuses the N > 1 arm's buffers
        dump_outputs(args.dump_outputs, *arm.outputs(got, offset), rank, world)
    total_ms = t_begin.elapsed_time(t_end)
    launches = codec.kernel_launches - launches0
    enc_ms = statistics.mean(s[0].elapsed_time(s[1]) for s in stats)
    dec_ms = statistics.mean(s[1].elapsed_time(s[2]) for s in stats)
    if dist is not None:
        t = torch.tensor([total_ms, enc_ms, dec_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, enc_ms, dec_ms = (float(v) for v in t.tolist())
        lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(lt)
        launches = int(lt.item())
    ms_step = total_ms / args.steps
    hist_ms = statistics.mean(s[3][0] for s in stats)
    host_ms = statistics.mean(s[3][1] for s in stats)
    pack_ms = statistics.mean(s[3][2] for s in stats)
    unpack_ms = statistics.mean(s[4][2] for s in stats)
    c_dec = c_local if world == 1 else arm.own_body  # compressed bytes this rank decodes
    peak, peak_src = peaks()

    def roof(label, kernels, alg_bytes, ms):
        ach = alg_bytes / 1e9 / (ms / 1e3) if ms > 0 else 0.0
        traffic = traffic_for(kernels) if (world == 1 and args.workload == "text-1G") else None
        return {"kernel": label, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "traffic_source": "profiles/traffic.json (committed ncu --set full capture, not measured in this run)"
                if traffic is not None else None,
                "algorithmic_bytes": alg_bytes, "ms": ms, "peak_source": peak_src}

    roofs = [roof("pack (region_bits_kernel + pack_runs_kernel)", ["region_bits_kernel", "pack_runs_kernel"], n + c_local, pack_ms),
             roof("unpack (region_sync_kernel + region_write_kernel)", ["region_sync_kernel", "region_write_kernel"],
                  c_dec + got, unpack_ms)]
    if world == 1:
        roofs.insert(0, roof("histogram_kernel", ["histogram_kernel"], n, hist_ms))
    dominant = max(roofs, key=lambda r: r["ms"])

    # ---- end to end with pinned HOST buffers (copies inside the timed region)
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, arm, inp, n, n_total, world, dist, barrier)

    configs = None
    if world == 1 and args.workload == "text-1G" and not args.no_configs:
        configs = run_other_configs(codec, stream, peak)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        k = min(n, CPU_SAMPLE)
        sample = inp[:k].cpu().numpy()
        te, td, which = time_oracle(sample)
        cpu = {"value": k / 1e9 / (te + td), "unit": "GB/s", "cores": 1, "kind": "port",
               "sample": f"first {k} B of {args.workload}, one encode + one decode; decode = {which}",
               "encode_gbs": k / 1e9 / te, "decode_gbs": k / 1e9 / td,
               "note": "C restatement of the reference algorithm; the Zig reference cannot be built here"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": n_total / 1e9 / (ms_step / 1e3), "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": args.workload, "bytes": n_total, "bytes_per_rank": n, "compressed_bytes_rank0": c_local,
                       "sharding": f"{world} contiguous byte ranges of one .et stream" if world > 1 else "none",
                       "sharded_path": getattr(arm, "path", None),
                       "l2": "inputs larger than L2 (126 MB), no explicit flush"},
            "encode_gbs": n_total / 1e9 / (enc_ms / 1e3), "decode_gbs": n_total / 1e9 / (dec_ms / 1e3),
            "encode_ms": enc_ms, "decode_ms": dec_ms,
            "stage_ms": {"histogram": hist_ms, "host_codebook": host_ms, "pack": pack_ms, "unpack": unpack_ms},
            "roofline": dominant, "rooflines": roofs,
            "encode_frac_of_hbm": (2 * n + c_local) / 1e9 / (enc_ms / 1e3) / peak,
            "decode_frac_of_hbm": (got + c_dec) / 1e9 / (dec_ms / 1e3) / peak,
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "verified_round_trip": verified,
            "decode_check_rounds": stats[-1][4][4], "clocks": clocks.summary(),
        }
        if numa:
            line["config"]["numa"] = numa
        if configs is not None:
            line["configs"] = configs
            base = [c for c in configs if c.get("workload") == "text-4G" and "round_trip_gbs" in c]
            if base:  # the one-GPU figure of the workload the N>1 runs shard: the denominator of strong scaling
                line["scale_base_gbs"] = base[0]["round_trip_gbs"]
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    codec.close()
    return 0


def run_e2e(args, arm, inp, n, n_total, world, dist, barrier):
    """The same step with pinned HOST buffers: N=1 through et_encode / et_decode (the reference-facing
    calls); N>1 pinned host -> device copy, the sharded device path, device -> pinned host copy."""
    import torch

    h_in, h_enc, h_dec = arm.e2e_buffers()
    steps = max(1, min(args.steps, 3))
    if world == 1:
        torch.from_numpy(h_in)[:] = inp[:n].cpu()
    else:
        h_in.copy_(inp[:n])
        h_dec[0].copy_(arm.range)
    times, h2d, d2h, got = [], 0, 0, 0
    for i in range(1 + steps):
        barrier()
        t0 = time.perf_counter()
        if world == 1:
            got, h2d, d2h = arm.e2e_step(h_in, h_enc, h_dec)
        else:
            got, h2d, d2h = arm.e2e_step(h_in, h_enc, h_dec, inp)
        barrier()
        if i >= 1:
            times.append(time.perf_counter() - t0)
    if world == 1:
        assert got == n and np.array_equal(h_dec[: 1 << 20], h_in[: 1 << 20])
    sec = statistics.mean(times)
    if dist is not None:
        t = torch.tensor([sec], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
        b = torch.tensor([h2d, d2h], dtype=torch.int64, device="cuda")
        dist.all_reduce(b)
        h2d, d2h = (int(v) for v in b.tolist())
    return {"value": n_total / 1e9 / sec, "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "steps": steps, "ms_per_step": sec * 1e3,
            "path": ("et_encode + et_decode (C ABI, pinned host buffers)" if world == 1 else
                     "pinned host -> device, sharded encode + decode (shard entry points of the C ABI), device -> pinned host")
                    + ", wall clock around the blocking calls"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--py-exchange", action="store_true", help="N>1: the exchanges in Python over torch.distributed instead of inside the library")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config block (text-5M, adversarial, text-4G)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path returned; --impl reference times a host sample")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload is None:
        args.workload = "text-1G" if max(world, args.gpus) == 1 else "text-4G"
    if args.impl == "reference":
        return run_reference(args, rank)
    if world != args.gpus:
        log(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE (launch N>1 under torch.distributed.run)")
    return run_ours(args, rank, world)


if __name__ == "__main__":
    sys.exit(main())
