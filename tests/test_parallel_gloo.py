"""world_size-2 tests (CPU) of the multi-GPU host logic -- over the library's own socket communicator and over a
gloo process group: probe partition and the single all-reduce of the sharded Hutchinson estimator.  The integrand is a stand-in with the same
protocol as `lanczos.integrand_spd` (callable + value_and_grad): the device path needs a GPU
and is covered by the `-m gpu` tests; here only the sharding / reduction plumbing is tested."""

import os
import socket
import subprocess
import sys
import textwrap

import numpy as np
import pytest
from conftest import ROOT

from experiments_lanczos_adjoints_b200 import parallel


@pytest.mark.parametrize("num,world", [(1024, 8), (10, 4), (3, 8), (0, 2), (7, 1)])
def test_shard_bounds_partition_exactly(num, world):
    blocks = [parallel.shard_bounds(num, r, world) for r in range(world)]
    assert blocks[0][0] == 0 and blocks[-1][1] == num
    for (lo, hi), (lo2, _) in zip(blocks, blocks[1:]):
        assert hi == lo2 and hi >= lo
    sizes = [hi - lo for lo, hi in blocks]
    assert max(sizes) - min(sizes) <= 1


@pytest.mark.parametrize("n,world", [(10, 2), (11, 4), (5, 8)])
def test_row_shard_index_work_covers_every_entry_once(n, world):
    """Row-sharded sparse operand: every COO entry lands in exactly one rank's A block and one
    rank's A^T block; local indices map back to the global ones (bit-exact host work)."""
    rng = np.random.default_rng(n)
    row, col = rng.integers(0, n, 40), rng.integers(0, n, 40)
    seen_a, seen_b = np.zeros(40, int), np.zeros(40, int)
    for r in range(world):
        chunk, idx_a, row_a, col_a, idx_b, row_b, col_b = parallel.shard_coo_rows(row, col, n, r, world)
        assert chunk * world >= n
        seen_a[idx_a] += 1
        seen_b[idx_b] += 1
        assert np.array_equal(row_a + r * chunk, row[idx_a]) and np.array_equal(col_a, col[idx_a])
        assert np.array_equal(row_b + r * chunk, col[idx_b]) and np.array_equal(col_b, row[idx_b])
        assert row_a.max(initial=0) < chunk and row_b.max(initial=0) < chunk
    assert np.all(seen_a == 1) and np.all(seen_b == 1)


WORKER_COMMON = """
    class Quadform:  # stand-in integrand: v^T diag(p) v, gradient v*v
        def __call__(self, v, p):
            return float(np.dot(v, p * v))
        def value_and_grad(self, v, p, want_dv0=True):
            return float(np.dot(v, p * v)), (None, v * v)

    rng = np.random.default_rng(0)
    probes = rng.integers(0, 2, size=(7, 5)) * 2.0 - 1.0   # odd count: ragged shards
    p = rng.uniform(1.0, 2.0, 5)
    est = parallel.hutchinson_sharded(Quadform(), lambda key: probes, group=group)
    ref = hutchinson.hutchinson(Quadform(), lambda key: probes)
    val = est(None, p)
    val2, (grad,) = est.value_and_grad(None, p)
    rval, (rgrad,) = ref.value_and_grad(None, p)
    assert np.allclose(val, rval) and np.allclose(val2, rval), (val, val2, rval)
    assert np.allclose(grad, rgrad), (grad, rgrad)
    # more ranks than probes: one rank has an empty shard and must issue the same collectives (ADVICE r1)
    one = probes[:1]
    est1 = parallel.hutchinson_sharded(Quadform(), lambda key: one, group=group)
    v1, (g1,) = est1.value_and_grad(None, p)
    assert np.allclose(v1, np.dot(one[0], p * one[0])) and np.allclose(g1, one[0] ** 2)
    # a sampler that generates by slice: the union over ranks does not depend on the number of ranks
    sampler = parallel.sharded_sampler(np.zeros(5), num=7)
    key = hutchinson.prng_key(3)
    full = sampler(key)
    lo, hi = parallel.shard_bounds(7, group.rank, group.world)
    assert np.array_equal(sampler.sample_slice(key, lo, hi), full[lo:hi]) and set(np.unique(full)) <= {-1.0, 1.0}
    est2 = parallel.hutchinson_sharded(Quadform(), sampler, group=group)
    ref2 = hutchinson.hutchinson(Quadform(), lambda k: full)
    assert np.allclose(est2(key, p), ref2(key, p))
    # host collectives of the communicator itself
    parts = group.allgather_bytes(bytes([group.rank]) * (group.rank + 1))
    assert parts == [bytes([r]) * (r + 1) for r in range(group.world)]
    assert np.allclose(group.allreduce_host(np.arange(3.0) + group.rank), 2 * np.arange(3.0) + 1)
    assert float(group.allreduce_host(np.array(float(group.rank)), op="max")) == 1.0
    group.barrier()
"""

WORKER = textwrap.dedent(
    """
    import os, sys
    import numpy as np
    sys.path.insert(0, os.environ["BL_ROOT"])
    from experiments_lanczos_adjoints_b200 import comm, parallel, hutchinson

    rank, world, _ = parallel.init_from_env()      # the library's own socket rendezvous: no torch
    assert world == 2 and "torch" not in sys.modules
    group = comm.default()
    """
) + textwrap.dedent(WORKER_COMMON) + textwrap.dedent(
    """
    comm.shutdown()
    assert "torch" not in sys.modules
    print("rank", rank, "ok")
    """
)

# The same estimator over a gloo process group: `group` only has to implement comm.Comm's host collectives, so a
# torch.distributed group plugs in through a ten-line adapter (kept in the tests: the package imports no torch).
WORKER_GLOO = textwrap.dedent(
    """
    import os, sys
    import numpy as np
    sys.path.insert(0, os.environ["BL_ROOT"])
    import torch, torch.distributed as dist
    from experiments_lanczos_adjoints_b200 import comm, parallel, hutchinson

    dist.init_process_group("gloo")

    class GlooComm(comm.Comm):
        rank, world, local_rank = dist.get_rank(), dist.get_world_size(), dist.get_rank()
        def allgather_bytes(self, payload):
            out = [None] * self.world
            dist.all_gather_object(out, bytes(payload))
            return out
        def allreduce_host(self, array, op="sum"):
            t = torch.from_numpy(np.array(array, dtype=np.float64, copy=True))
            dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
            return t.numpy()
        def barrier(self):
            dist.barrier()

    group = GlooComm()
    rank = group.rank
    assert group.world == 2
    """
) + textwrap.dedent(WORKER_COMMON) + textwrap.dedent(
    """
    dist.destroy_process_group()
    print("rank", rank, "ok")
    """
)


@pytest.mark.parametrize("worker", ["sockets", "gloo"])
def test_sharded_hutchinson_matches_single_process(tmp_path, worker):
    script = tmp_path / "worker.py"
    script.write_text(WORKER if worker == "sockets" else WORKER_GLOO)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    # host logic only: with a device visible, `comm.init_from_env` binds GPU LOCAL_RANK, which a machine with one
    # GPU does not have for rank 1; hidden devices make the run the same on machines with none, one or several GPUs
    env = dict(os.environ, BL_ROOT=ROOT, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2",
               CUDA_VISIBLE_DEVICES="")  # fmt: skip
    procs = [
        subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)),
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        for r in range(2)
    ]  # fmt: skip
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, out) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, out
        assert f"rank {r} ok" in out


def test_package_and_bench_import_no_torch():
    """north_star: host code reaches CUDA only through the C ABI, with no PyTorch.  The package and bench.py must
    not import torch on any path (the multi-GPU layer uses comm.py + bl_dist_nccl_*)."""
    import re

    offenders = []
    for base, _dirs, files in os.walk(os.path.join(ROOT, "experiments_lanczos_adjoints_b200")):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(base, f)).read()
                if re.search(r"^\s*(import torch|from torch)", text, flags=re.M):
                    offenders.append(f)
    text = open(os.path.join(ROOT, "bench.py")).read()
    if re.search(r"^\s*(import torch|from torch)", text, flags=re.M):
        offenders.append("bench.py")
    assert not offenders, offenders
