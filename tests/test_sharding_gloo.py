"""CPU test of the N>1 path (world_size 2, gloo): reads sharded over ranks, target broadcast once,
distances gathered on rank 0 -- the same plumbing bench.py uses over NCCL.  Each rank aligns its
shard with the host emulation of the kernels (no GPU here); rank 0 compares the gathered vector
with the single-process result."""
import os
import subprocess
import sys

from edlib_b200._ffi import REPO

WORKER = r'''
import os, sys
sys.path.insert(0, %(repo)r); sys.path.insert(0, os.path.join(%(repo)r, "tests"))
import numpy as np, torch, torch.distributed as dist
from edlib_b200 import sharding, workloads
from edlib_b200._ffi import EdlibLib
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
lib = EdlibLib(os.path.join(%(repo)r, "tests", "emul", "libedlib_emul.so"), has_batch=True)
N, TL = 301, 20000
target = workloads.random_dna(TL, 1) if rank == 0 else None
target = sharding.broadcast_target(target, TL, torch.device("cpu"))
_, reads = workloads.reads_vs_target(N, 150, TL, seed=9)           # every rank can regenerate the seeded batch
lo, hi = sharding.shard_range(N, rank, world)
t = target.tobytes()
st, res = lib.align_batch([reads[i].tobytes() for i in range(lo, hi)], [t] * (hi - lo), -1, 2, 0)
assert st == 0
eds = np.array([r["editDistance"] for r in res], dtype=np.int32)
got = sharding.gather_int32(eds, torch.device("cpu"))
# the variants bench.py's strong-scaling step uses: target into a caller buffer, gather with known counts
tbuf = np.zeros(TL, dtype=np.uint8)
sharding.broadcast_target_into(target if rank == 0 else None, tbuf, torch.device("cpu"))
assert (tbuf == target).all()
counts = [sharding.shard_range(N, r, world)[1] - sharding.shard_range(N, r, world)[0] for r in range(world)]
got2 = sharding.gather_int32_known(eds, counts, torch.device("cpu"))
if rank == 0:
    assert got2.tolist() == got.tolist()
    st, full = lib.align_batch([reads[i].tobytes() for i in range(N)], [t] * N, -1, 2, 0)
    assert got.tolist() == [r["editDistance"] for r in full]
    print("GLOO_OK", len(got))
dist.destroy_process_group()
'''


def test_two_rank_shard_broadcast_gather(tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(REPO, "tests", "emul")], check=True)
    subprocess.run(["make", "-s", "-C", os.path.join(REPO, "edlib_b200", "csrc"), "../lib/libsynth.so"], check=True)
    script = str(tmp_path / "edlib_gloo_worker.py")
    with open(script, "w") as f:
        f.write(WORKER % {"repo": REPO})
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29577", script],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    assert "GLOO_OK 301" in out.stdout


def test_shard_ranges_cover_everything():
    from edlib_b200.sharding import shard_range
    for n in (0, 1, 7, 1000001):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1
