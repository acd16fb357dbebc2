"""Regenerates tests/golden/ from the reference's own fixtures.

    python tests/golden/make_golden.py <typio/entreepy checkout>/res

Inputs : res/*.txt of typio/entreepy (the files test.zig:35-72 round-trips; public-domain text).
Outputs: <name>            the input bytes (test DATA, not reference source code)
         <name>.et         .et file produced by the CPU oracle (oracle/entreepy_oracle.c)
         manifest.json     sizes, sha256s, header lengths, code-length summary, Midsummer histogram
The tests need no copy of the reference: the inputs are committed here.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import oracle  # noqa: E402

if len(sys.argv) != 2:
    sys.exit(__doc__)
RES = sys.argv[1]
NAMES = ["test.txt", "nice.shakespeare.txt", "a_midsummer_nights_dream.txt"]

# SURVEY.md §8c — derived by an independent restatement during the survey.
SURVEY = {
    "test.txt": (42, 26, "761b5bc3dcb9d8487eaa764b7c1b207774caff78a464b229c56f939417af764d"),
    "nice.shakespeare.txt": (374, 109, "795f27fd81733435fbaa1e58d260950eec57f800652245464b7e3209407a2409"),
    "a_midsummer_nights_dream.txt": (66312, 311, "d152197f8c5ee87c68ca812929ebc92ffd74b0fecbdd6c491b203d19479eb97b"),
}

manifest = {}
for name in NAMES:
    data = open(os.path.join(RES, name), "rb").read()
    et = oracle.encode(data).tobytes()
    occ = oracle.histogram(data)
    _, lens = oracle.build_dictionary(occ)
    body_bits = int(sum(int(occ[s]) * int(lens[s]) for s in range(256)))
    header = len(et) - (body_bits + 7) // 8
    size, hdr, sha = SURVEY[name]
    assert (len(et), header, hashlib.sha256(et).hexdigest()) == (size, hdr, sha), name
    shutil.copyfile(os.path.join(RES, name), os.path.join(HERE, name))
    open(os.path.join(HERE, name + ".et"), "wb").write(et)
    manifest[name] = {
        "n": len(data),
        "sha256": hashlib.sha256(data).hexdigest(),
        "et_bytes": len(et),
        "et_header_bytes": header,
        "et_sha256": sha,
        "body_bits": body_bits,
        "min_len": int(min(l for l in lens if l)),
        "max_len": int(max(lens)),
        "distinct": int((occ > 0).sum()),
    }
    if name == "a_midsummer_nights_dream.txt":
        manifest["midsummer_histogram"] = [int(c) for c in occ]
json.dump(manifest, open(os.path.join(HERE, "manifest.json"), "w"), indent=1)
print(json.dumps({k: v for k, v in manifest.items() if k != "midsummer_histogram"}, indent=1))
