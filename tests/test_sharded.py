"""Multi-process tests of the sharded build (SURVEY.md 8e).

CPU (gloo, world_size 2 and 3): shard ranges, unique-id broadcast and assembly of rank-local exports,
with the device emulated by the C oracle.  GPU (nccl, needs >= 2 GPUs): the real collective build,
bit-exact against the oracle's build of the whole read set."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from tests.helpers import ROOT


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run(world, *worker_args, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "sharded_worker.py")] + list(worker_args)
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert res.returncode == 0 and "SHARDED_PARITY OK" in res.stdout, (res.stdout[-3000:], res.stderr[-3000:])


def test_shard_ranges_partition_the_reads():
    from amira_b200 import sharded
    for n in (0, 1, 7, 1000, 1001):
        for world in (1, 2, 3, 8):
            r = [sharded.shard_range(n, i, world) for i in range(world)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(r, r[1:]))
            sizes = [b - a for a, b in r]
            assert max(sizes) - min(sizes) <= 1


def test_assemble_is_identity_for_one_rank():
    from amira_b200 import sharded, synth
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 500)
    a = c_oracle.COracleGraph(ids, off, 3).arrays()
    assert O.diff_arrays(sharded.assemble_arrays([a]), a) == []


@pytest.mark.parametrize("world,args", [(2, ("--k", "3", "--reads", "4000")),
                                        (3, ("--k", "5", "--reads", "3000", "--positions")),
                                        (2, ("--k", "3", "--reads", "2000", "--uneven"))])
def test_sharded_host_logic_gloo(world, args):
    _run(world, "--backend", "gloo", *args)


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.parametrize("args", [("--config", "c3", "--k", "3", "--reads", "60000"),
                                  ("--config", "c5", "--k", "5", "--reads", "40000", "--positions"),
                                  ("--config", "c2", "--k", "3", "--reads", "3000", "--uneven"),
                                  ("--config", "c4", "--k", "7", "--reads", "50000"),
                                  ("--config", "c3", "--k", "1", "--reads", "3000")])
def test_sharded_build_matches_oracle_nccl(args):
    n = _n_gpus()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    _run(min(n, 8) if "--uneven" not in args else 2, "--backend", "nccl", *args)
