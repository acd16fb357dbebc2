import os, sys, time, json
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch, torch.distributed as dist
import entreepy_b200 as et
from entreepy_b200 import sharded, synth
local = int(os.environ["LOCAL_RANK"]); torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rank, world = dist.get_rank(), dist.get_world_size()
codec = et.Codec(local)
n_total = (1 << 32) - 16
plan = sharded.ShardPlan(n_total, world, rank)
man = json.load(open(os.path.join(ROOT, "tests/golden/manifest.json")))
thr = synth.thresholds_from_weights(synth.text_weights(man["midsummer_histogram"]))
inp = torch.empty(plan.n_local + 16, dtype=torch.uint8, device="cuda")
stream = torch.cuda.current_stream().cuda_stream
codec.synth_dev(inp.data_ptr(), plan.n_local, synth.SEED, plan.lo, thr)
be = sharded.GpuBackend(codec, stream)
comm = sharded.Comm(dist, torch.device("cuda"))
coder = sharded.ShardedCodec(be, plan, comm)
body = torch.empty(plan.n_local + 16384, dtype=torch.uint8, device="cuda")
# wrap phases
import types
T = {}
def timed(name, fn):
    def w(*a, **k):
        torch.cuda.synchronize(); t0 = time.perf_counter(); r = fn(*a, **k); torch.cuda.synchronize(); T[name] = T.get(name, 0) + time.perf_counter() - t0; return r
    return w
be.histogram = timed("histogram", be.histogram)
be.head_symbols = timed("head_symbols", be.head_symbols)
be.pack_shard = timed("pack_shard", be.pack_shard)
be.unpack_shard = timed("unpack_shard", be.unpack_shard)
be.or_byte = timed("or_byte", be.or_byte)
comm.allgather_ints = timed("allgather_ints", comm.allgather_ints)
sharded.build_codebook = timed("build_codebook", sharded.build_codebook)
sharded.write_header = timed("write_header", sharded.write_header)
sharded.parse_header = timed("parse_header", sharded.parse_header)
be.shard_bits = timed("shard_bits", be.shard_bits)
for it in range(6):
    if it == 1: T.clear(); tenc = tdec = 0
    dist.barrier(); torch.cuda.synchronize(); t0 = time.perf_counter()
    res = coder.encode(inp, body)
    torch.cuda.synchronize(); t1 = time.perf_counter()
    if it == 0:
        rng = coder.scatter_body(res, body).clone()
        dec = torch.empty(int(n_total / world * 1.25) + (1 << 20), dtype=torch.uint8, device="cuda")
    dist.barrier(); torch.cuda.synchronize(); t2 = time.perf_counter()
    d = coder.decode(res.header[4:], res.body_bytes, rng, dec)
    torch.cuda.synchronize(); t3 = time.perf_counter()
    if it: tenc += t1 - t0; tdec += t3 - t2
if rank == 0:
    print("encode ms", tenc / 5 * 1e3, "decode ms", tdec / 5 * 1e3)
    for k, v in sorted(T.items(), key=lambda x: -x[1]): print(f"  {k:16s} {v / 5 * 1e3:8.3f} ms/step")
    print("cpus usable by a rank:", len(os.sched_getaffinity(0)), "of", os.cpu_count())
# every rank: its own phase times (skew shows up as waiting inside the exchanges)
line = f"rank {rank}: enc {tenc / 5 * 1e3:.3f} dec {tdec / 5 * 1e3:.3f} | " + " ".join(
    f"{k}={v / 5 * 1e3:.3f}" for k, v in sorted(T.items()) if k in ("histogram", "pack_shard", "unpack_shard", "allgather_ints"))
for r in range(world):
    dist.barrier()
    if r == rank:
        print(line, flush=True)
dist.destroy_process_group()
