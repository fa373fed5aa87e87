"""Worker of the sharded refusal test of amira_gmg_gene_paths (launched with torch.distributed.run, one process and one
GPU per rank): after a collective build it must return AMIRA_E_STATE on every rank.  Prints SHARDED_GENE_PATHS OK on
rank 0."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    from amira_b200 import _lib, sharded, synth
    from amira_b200.device_graph import DeviceGraph
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl")
    g = DeviceGraph(rank)
    uid = [g.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    g.comm_init(uid[0], rank, world)
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 2000)
    lo, hi = sharded.shard_range(len(off) - 1, rank, world)
    sub_off = off[lo:hi + 1] - off[lo]
    g.build(ids[off[lo]:off[hi]].copy(), sub_off.copy(), 3)
    r = (C.c_int32 * 1)(1)
    status = g._lib.amira_gmg_gene_paths(g._h, r, 1, C.byref(C.c_int64()), *[None] * 14)
    assert status == _lib.E_STATE, (status, _lib.last_error())
    dist.barrier()
    if rank == 0:
        print("SHARDED_GENE_PATHS OK", flush=True)
    g.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
