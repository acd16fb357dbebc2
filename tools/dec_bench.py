"""Decode (and encode) timing of one synthetic stream through the C ABI, device resident (developer tool, run under gpurun).

    python tools/dec_bench.py [log2_bytes=30] [reps=10] [kind=text|fib|u255]
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import entreepy_b200 as et  # noqa: E402
from entreepy_b200 import synth  # noqa: E402

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 30
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
kind = sys.argv[3] if len(sys.argv) > 3 else "text"
n = 1 << lg
man = json.load(open(os.path.join(ROOT, "tests/golden/manifest.json")))
if kind == "text":
    w = synth.text_weights(man["midsummer_histogram"])
elif kind == "fib":
    w = synth.fibonacci_weights(32)
else:
    w = [0] + [1] * 255
thr = synth.thresholds_from_weights(w)
c = et.Codec(0)
if os.environ.get("ET_LANE_MIN_BYTES"):
    c.set_tuning(et._abi.TUNE_LANE_MIN_BYTES, int(os.environ["ET_LANE_MIN_BYTES"]))
dev = torch.empty(n, dtype=torch.uint8, device="cuda")
c.synth_dev(dev.data_ptr(), n, synth.SEED, 0, thr)
enc = torch.empty(n + n // 8 + 16384, dtype=torch.uint8, device="cuda")
dec = torch.zeros(n, dtype=torch.uint8, device="cuda")
size = c.encode_dev(dev.data_ptr(), n, enc.data_ptr(), enc.numel())


def timed(fn):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(min(ts))


e_med, e_min = timed(lambda: c.encode_dev(dev.data_ptr(), n, enc.data_ptr(), enc.numel()))
d_med, d_min = timed(lambda: c.decode_dev(enc.data_ptr() + 4, size - 4, dec.data_ptr(), n))
ok = bool(torch.equal(dec, dev))
print(json.dumps({"kind": kind, "n": n, "et_bytes": size, "encode_ms": e_med, "encode_min_ms": e_min, "decode_ms": d_med,
                  "decode_min_ms": d_min, "encode_gbs": n / e_med / 1e6, "decode_gbs": n / d_med / 1e6, "round_trip_ok": ok,
                  "rounds": c.last_decode_rounds}))
c.close()
