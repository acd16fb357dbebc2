"""Small round trips through the lane-run pack and the lane-interleaved decoder, for compute-sanitizer
(developer tool, run under gpurun:  compute-sanitizer --tool memcheck python tests/dev/sanitize_small.py)."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
os.environ.setdefault("ET_LANE_MIN_BYTES", "0")
import entreepy_b200 as et  # noqa: E402
from entreepy_b200 import synth  # noqa: E402
from oracle import oracle  # noqa: E402

man = json.load(open(os.path.join(ROOT, "tests/golden/manifest.json")))
thr = synth.thresholds_from_weights(synth.text_weights(man["midsummer_histogram"]))
host = synth.generate(300000, thr)
rng = np.random.default_rng(3)
with et.Codec(0) as c:
    for n in (30011, 100003, 300000):
        data = host[:n]
        m, enc = c.encode(data, et.EncodeFlags(write_output=True, no_scratch_limit=True))
        assert enc.tobytes() == oracle.encode(data, cap=9000 + 5 * n).tobytes(), n
        k, dec = c.decode(enc[4:m])
        assert k == n and dec.tobytes() == data.tobytes(), n
    w = rng.random(256) ** 8
    data = rng.choice(256, 200000, p=w / w.sum()).astype(np.uint8)
    m, enc = c.encode(data, et.EncodeFlags(write_output=True, no_scratch_limit=True))
    want = oracle.encode(data, cap=9000 + 5 * data.size).tobytes()
    assert enc.tobytes() == want
    k, dec = c.decode(enc[4:m])
    assert dec.tobytes() == oracle.decode(want[4:], data.size).tobytes()
    # slowly synchronising code (transfer functions)
    data = rng.integers(1, 256, 150001, dtype=np.uint8)
    m, enc = c.encode(data, et.EncodeFlags(write_output=True, no_scratch_limit=True))
    k, dec = c.decode(enc[4:m])
    assert k == data.size and dec.tobytes() == data.tobytes()
print("sanitize_small ok")
