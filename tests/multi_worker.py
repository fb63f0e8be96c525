"""Worker of the multi-rank tests (launched with torch.distributed.run, one process per rank).

    python -m torch.distributed.run --nproc-per-node N tests/multi_worker.py <mode> <out_dir>

mode = cpu : gloo only; checks the host-side sharding logic (no GPU).
mode = gpu : every rank runs its row shard of every case through the engine and saves its result rows; the parent test
             compares the union over the ranks with the oracle.  Cases (tests/test_multi_rank.py builds the same tables):
               spread : rows shuffled over the ranks -> optimistic partition + peer pull (no histogram pass, no NCCL
                        exchange; asserted through phase_ms)
               skewed : two long connections sit on the last rank -> a slot overflows there, every rank falls back to
                        the exact partition, which the peers pull as well (no receive buffer)
               xpull  : the skewed table on a fresh engine, two runs per algorithm (second engine)
               nccl   : the spread table with the peer pull switched off: exact partition + NCCL all-to-all (chunked,
                        overlapped) (third engine)
               ncclskew : the skewed table on the third engine: the NCCL exchange with the spill path behind it"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from theia_b200 import sharding, synth  # noqa: E402


def case_table(name):
    table = synth.make_flows(4000, 40, seed=77, dup_frac=0.05, ragged=True)      # same table on every rank
    if name == "skewed":
        t2 = synth.make_flows(2, 6000, seed=78)                                  # two long connections -> spill path
        table = {k: np.concatenate([table[k], t2[k]]) for k in table}
    else:
        t2 = synth.make_flows(3, 900, seed=79)                                   # long, but spread over the ranks
        table = {k: np.concatenate([table[k], t2[k]]) for k in table}
        perm = np.random.default_rng(5).permutation(len(table["value"]))
        table = {k: v[perm] for k, v in table.items()}
    return table


def main():
    mode, out_dir = sys.argv[1], sys.argv[2]
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group("gloo")
    for name in ("spread", "skewed"):
        table = case_table(name)
        total = len(table["value"])
        mine = sharding.shard_rows(table, rank, world)
        own = sharding.owner_rank(table, world, total)
        expect_owned = int((own == rank).sum())
        counts = [None] * world
        dist.all_gather_object(counts, (len(mine["value"]), expect_owned))
        assert sum(c[0] for c in counts) == total and sum(c[1] for c in counts) == total
        # a connection has exactly one owner
        h = sharding.key_hash(table)
        order = np.argsort(h, kind="stable")
        same = h[order][1:] == h[order][:-1]
        assert (own[order][1:][same] == own[order][:-1][same]).all()
    if mode == "gpu":
        from theia_b200.engine import TadEngine
        os.environ["TAD_EXCHANGE_MIN_ROWS"] = "0"        # exercise the chunked (overlapped) exchange on these small tables
        local = int(os.environ.get("LOCAL_RANK", rank))

        def engine(peer_pull):
            os.environ["TAD_PEER_PULL"] = "1" if peer_pull else "0"
            uid = [TadEngine.get_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            return TadEngine(device=local, world_size=world, rank=rank, nccl_unique_id=uid[0])

        eng = engine(True)
        for rep in range(2):                              # the second round reuses the mapped buffers (steady state)
            for name in ("spread", "skewed", "spread"):
                table = case_table(name)
                total = len(table["value"])
                mine = sharding.shard_rows(table, rank, world)
                expect_owned = int((sharding.owner_rank(table, world, total) == rank).sum())
                for algo in ("EWMA", "DBSCAN"):
                    # global_rows: given by the host in the first round, agreed on by the ranks in the second
                    got, st = eng.run(mine, algo=algo, tad_id="multi", emit_all=True, global_rows=total if rep == 0 else 0)
                    assert st["rows_owned"] == expect_owned, (rank, name, st["rows_owned"], expect_owned)
                    assert st["rows_kept"] == len(mine["value"]), (rank, name, st["rows_kept"], len(mine["value"]))
                    optimistic = st["phase_ms"]["hist"] == 0.0
                    assert optimistic == (name == "spread"), (rank, name, st["phase_ms"])
                    np.savez(os.path.join(out_dir, "res_%s_%s_%d.npz" % (name, algo, rank)), **got)
        eng.close()
        # the exact partition pulled by the peers (no receive buffer): the skewed table overflows a slot, every rank falls back
        eng = engine(True)
        table = case_table("skewed")
        total = len(table["value"])
        mine = sharding.shard_rows(table, rank, world)
        for algo in ("EWMA", "DBSCAN"):
            for rep in range(2):
                got, st = eng.run(mine, algo=algo, tad_id="multi", emit_all=True, global_rows=total)
            assert st["phase_ms"]["hist"] > 0.0 and st["rows_kept"] == len(mine["value"])
            np.savez(os.path.join(out_dir, "res_xpull_%s_%d.npz" % (algo, rank)), **got)
        eng.close()
        eng = engine(False)
        table = case_table("spread")
        mine = sharding.shard_rows(table, rank, world)
        got, st = eng.run(mine, algo="EWMA", tad_id="multi", emit_all=True, global_rows=len(table["value"]))
        assert st["phase_ms"]["hist"] > 0.0
        np.savez(os.path.join(out_dir, "res_nccl_EWMA_%d.npz" % rank), **got)
        table = case_table("skewed")                                       # the NCCL exchange with the spill path behind it
        mine = sharding.shard_rows(table, rank, world)
        got, st = eng.run(mine, algo="EWMA", tad_id="multi", emit_all=True, global_rows=len(table["value"]))
        np.savez(os.path.join(out_dir, "res_ncclskew_EWMA_%d.npz" % rank), **got)
        eng.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
