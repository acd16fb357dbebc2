"""Batched against per-stream device decode and encode of many .et streams (developer tool; needs a B200).

    python tools/batch_bench.py [--reps 7] [--json FILE] [--only decode|encode]

Text-distribution streams are generated on the device (et_synth_dev) and encoded (et_encode_dev).  For every batch size B
in {1, 16, 256, 2048} and stream size in {4 KiB, 64 KiB, 1 MiB}, and for one mixed batch (255 streams of 64 KiB, one of
64 MiB and one of bytes uniform over 1..255, the last two taken by the per-stream decoders), decode is timed with CUDA events after a
warm-up, alternating in the same process:
  batch  one et_decode_batch_dev call over the B streams;
  loop   a Python loop of et_decode_dev over the same streams.
Every output is compared with the original before the cell's times are reported.  Rates are uncompressed bytes over the
median time; launches are kernel launches per call (et_ctx_kernel_launches).  The card's name and power limit come first.

Encode cells ("enc ..."): the same sizes, and a mixed batch of 255 texts of 64 KiB, one of 256 MiB (encoded one by one,
as et_encode_dev does it) and one of uniform bytes:
  batch  one et_encode_batch_dev call over the B texts;
  loop   a Python loop of et_encode_dev over the same texts.
Before the times are reported, the statuses, sizes and every output byte of the batch are compared with the loop's.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import entreepy_b200 as et  # noqa: E402
from entreepy_b200 import _abi, synth  # noqa: E402

WRITE = _abi.FLAG_WRITE_OUTPUT


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        power = r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


class Streams:
    """Encoded streams on the device: the originals side by side in `text`, the decoded copies go to `out`."""

    def __init__(self, codec, pieces):
        # pieces: [(size, thresholds, seed)]
        self.sizes = [p[0] for p in pieces]
        offs = np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int64)
        self.text = torch.empty(int(offs[-1]), dtype=torch.uint8, device="cuda")
        self.out = torch.zeros_like(self.text)
        caps = [s + s // 4 + 8192 for s in self.sizes]
        eoffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.int64)
        self.enc = torch.empty(int(eoffs[-1]), dtype=torch.uint8, device="cuda")
        self.items = []
        for k, (size, thr, seed) in enumerate(pieces):
            codec.synth_dev(self.text.data_ptr() + int(offs[k]), size, seed, int(offs[k]), thr)
            n = codec.encode_dev(self.text.data_ptr() + int(offs[k]), size, self.enc.data_ptr() + int(eoffs[k]), caps[k],
                                 WRITE | _abi.FLAG_NO_SCRATCH_LIMIT)
            self.items.append((self.enc.data_ptr() + int(eoffs[k]) + 4, n - 4, self.out.data_ptr() + int(offs[k]), size))
        self.offs = offs

    def verify(self, b):
        torch.cuda.synchronize()
        end = int(self.offs[b])
        return bool(torch.equal(self.out[:end], self.text[:end]))


def run_cell(codec, streams, b, reps, label):
    items = streams.items[:b]
    total = int(streams.offs[b])

    def batch():
        res = codec.decode_batch_dev(items)
        assert all(r == (_abi.OK, it[3]) for r, it in zip(res, items)), label

    def loop():
        for d_in, n, d_out, cap in items:
            codec.decode_dev(d_in, n, d_out, cap)

    out = {"cell": label, "streams": b, "bytes": total}
    for name, fn in (("batch", batch), ("loop", loop)):
        streams.out.zero_()
        torch.cuda.synchronize()  # the library's stream does not wait for torch's
        before = codec.kernel_launches
        fn()  # warm-up, and the output that is checked
        out[f"{name}_launches"] = codec.kernel_launches - before
        if not streams.verify(b):
            raise SystemExit(f"{label}: {name} decode differs from the original")
    times = {"batch": [], "loop": []}
    for _ in range(reps):
        for name, fn in (("batch", batch), ("loop", loop)):
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn()
            z.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(z))
    for name in ("batch", "loop"):
        ms = float(np.median(times[name]))
        out[f"{name}_ms"] = round(ms, 4)
        out[f"{name}_gbs"] = round(total / ms / 1e6, 3)
    out["loop_over_batch"] = round(out["loop_ms"] / out["batch_ms"], 2)
    streams.out.zero_()
    torch.cuda.synchronize()
    batch()
    if not streams.verify(b):  # the timed calls wrote the same text
        raise SystemExit(f"{label}: batch decode differs from the original after timing")
    return out


class Texts:
    """Texts side by side on the device, and two output buffers (batch, loop) with room for each one's .et file."""

    def __init__(self, codec, pieces):
        self.sizes = [p[0] for p in pieces]
        offs = np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int64)
        self.text = torch.empty(int(offs[-1]), dtype=torch.uint8, device="cuda")
        for k, (size, thr, seed) in enumerate(pieces):
            codec.synth_dev(self.text.data_ptr() + int(offs[k]), size, seed, int(offs[k]), thr)
        caps = [s + s // 4 + 8192 for s in self.sizes]
        self.eoffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.int64)
        self.out = {name: torch.zeros(int(self.eoffs[-1]), dtype=torch.uint8, device="cuda") for name in ("batch", "loop")}
        self.items = {name: [(self.text.data_ptr() + int(offs[k]), self.sizes[k], buf.data_ptr() + int(self.eoffs[k]), caps[k])
                             for k in range(len(pieces))] for name, buf in self.out.items()}
        self.offs = offs


def run_encode_cell(codec, texts, b, reps, label):
    total = int(texts.offs[b])
    flags = WRITE | _abi.FLAG_NO_SCRATCH_LIMIT
    results = {}

    def batch():
        results["batch"] = codec.encode_batch_dev(texts.items["batch"][:b], flags)

    def loop():
        results["loop"] = [(_abi.OK, codec.encode_dev(d_in, n, d_out, cap, flags)) for d_in, n, d_out, cap in texts.items["loop"][:b]]

    out = {"cell": label, "streams": b, "bytes": total}
    for name, fn in (("batch", batch), ("loop", loop)):
        texts.out[name].zero_()
        torch.cuda.synchronize()  # the library's stream does not wait for torch's
        before = codec.kernel_launches
        fn()  # warm-up, and the output that is checked
        out[f"{name}_launches"] = codec.kernel_launches - before
    torch.cuda.synchronize()
    end = int(texts.eoffs[b])
    if results["batch"] != results["loop"] or not torch.equal(texts.out["batch"][:end], texts.out["loop"][:end]):
        raise SystemExit(f"{label}: batch encode differs from the single calls")
    times = {"batch": [], "loop": []}
    for _ in range(reps):
        for name, fn in (("batch", batch), ("loop", loop)):
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn()
            z.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(z))
    for name in ("batch", "loop"):
        ms = float(np.median(times[name]))
        out[f"{name}_ms"] = round(ms, 4)
        out[f"{name}_gbs"] = round(total / ms / 1e6, 3)
    out["loop_over_batch"] = round(out["loop_ms"] / out["batch_ms"], 2)
    out["encoded_bytes"] = int(sum(r[1] for r in results["batch"]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--json", default=None, help="also write the results here")
    ap.add_argument("--only", choices=("decode", "encode"), default=None, help="run only the decode or the encode cells")
    args = ap.parse_args()
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}))
    man = json.load(open(os.path.join(ROOT, "tests", "golden", "manifest.json")))
    text = synth.thresholds_from_weights(synth.text_weights(man["midsummer_histogram"]))
    # the decode cell checks its text against the original: the 255-symbol variant, since with all 256 byte values the
    # format drops a symbol (DESIGN.md §0); the encode cell compares the batch with the loop, so it keeps all 256
    uniform255 = synth.thresholds_from_weights(synth.uniform_weights(1))
    uniform = synth.thresholds_from_weights(synth.uniform_weights())
    codec = et.Codec(0)
    results = []
    for size in (4 << 10, 64 << 10, 1 << 20) if args.only != "encode" else ():
        streams = Streams(codec, [(size, text, synth.SEED)] * 2048)
        for b in (1, 16, 256, 2048):
            r = run_cell(codec, streams, b, args.reps, f"{b}x{size >> 10}KiB")
            print(json.dumps(r), flush=True)
            results.append(r)
        del streams
        torch.cuda.empty_cache()
    if args.only != "encode":
        mixed = Streams(codec, [(64 << 10, text, synth.SEED)] * 255 + [(64 << 20, text, synth.SEED), (1 << 20, uniform255, synth.SEED)])
        r = run_cell(codec, mixed, 257, args.reps, "mixed: 255x64KiB + 64MiB text + 1MiB uniform")
        print(json.dumps(r), flush=True)
        results.append(r)
        del mixed
        torch.cuda.empty_cache()
    if args.only != "decode":
        for size in (4 << 10, 64 << 10, 1 << 20):
            texts = Texts(codec, [(size, text, synth.SEED)] * 2048)
            for b in (1, 16, 256, 2048):
                r = run_encode_cell(codec, texts, b, args.reps, f"enc {b}x{size >> 10}KiB")
                print(json.dumps(r), flush=True)
                results.append(r)
            del texts
            torch.cuda.empty_cache()
        mixed = Texts(codec, [(64 << 10, text, synth.SEED)] * 255 + [(256 << 20, text, synth.SEED), (1 << 20, uniform, synth.SEED)])
        r = run_encode_cell(codec, mixed, 257, args.reps, "enc mixed: 255x64KiB + 256MiB text + 1MiB uniform")
        print(json.dumps(r), flush=True)
        results.append(r)
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"card": name, "power_limit": power, "results": results}, f, indent=1)
    codec.close()


if __name__ == "__main__":
    main()
