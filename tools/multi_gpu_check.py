#!/usr/bin/env python
"""Run under torchrun (one rank per GPU): sharded recruitment == the CPU oracle on the whole read set.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tools/multi_gpu_check.py

Checks (rank 0): identical rare set, identical edge set, identical unique k-mers, identical increment count; every
rank: its own clouds equal the oracle's clouds of its reads.  Test infrastructure (uses oracle/)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from centroflye_b200 import synth
    from centroflye_b200.dist import ShardedRecruiter
    from centroflye_b200.engine import Engine, band_to_int
    from centroflye_b200.ingest import batch_from_synth
    from oracle import c_oracle

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    eng = Engine(f"cuda:{local}")
    unit = synth.hor_unit(4, 60, 0.25, seed=5)
    genome, a0, alen = synth.simulate_genome(unit, 160, 0.02, 6, flank_len=2000)
    kw = dict(median_len=7000, sigma=0.4, min_len=5200, max_len=20000)
    reads = synth.simulate_reads(genome, a0, alen, unit, 20, 0.05, 7, **kw)
    mine = synth.simulate_reads(genome, a0, alen, unit, 20, 0.05, 7, shard=(rank, world), **kw)
    all_ids = {r.r_id for r in reads}
    assert all(r.r_id in all_ids for r in mine), "shard holds a read that is not in the whole set"
    n_mine = torch.tensor([len(mine)], dtype=torch.int64, device=f"cuda:{local}")
    dist.all_reduce(n_mine)
    assert int(n_mine.item()) == len(reads), "shards do not partition the read set"
    k, max_nonuniq, min_d, max_d, min_cov = 19, 3, 1, 150, 4
    lo, hi = band_to_int(0.9 * 20 * 0.4, 3.0 * 20 * 0.4)
    batch, units = batch_from_synth(mine, len(unit))
    rec = ShardedRecruiter(eng, batch, units, k, rank, world)
    eng.docfreq_mode = "resident"  # the table-based exchanges: the full all-to-all of table records ...
    rec.nominate = False
    index_full, _, _ = rec.step(lo, hi, max_nonuniq, min_d, max_d, min_cov)
    full_bytes, rec.bytes_exchanged = rec.bytes_exchanged, 0
    rec.nominate = True   # ... and nominate-then-sum give the same rare set
    index_nom, _, _ = rec.step(lo, hi, max_nonuniq, min_d, max_d, min_cov)
    assert np.array_equal(index_nom.sorted_keys.cpu().numpy(), index_full.sorted_keys.cpu().numpy()), "the two table exchanges disagree"
    assert rec.bytes_exchanged < full_bytes
    eng.docfreq_mode = "stream"    # the default: all-to-all of phase 1's records, phase 2 on the owned partitions
    rec.bytes_exchanged = 0
    for _ in range(2):  # the second step runs with the adapted partition grouping / buffer sizes
        index, csr, res = rec.step(lo, hi, max_nonuniq, min_d, max_d, min_cov)
    keys = index.sorted_keys.cpu().numpy().view(np.uint64)
    assert eng.stream_fallbacks == 0, "the record exchange fell back"
    assert np.array_equal(keys, index_full.sorted_keys.cpu().numpy().view(np.uint64)), "record exchange != table exchange"

    whole_batch, whole_units = batch_from_synth(reads, len(unit))
    want = c_oracle.recruit(whole_batch, whole_units, k, lo, hi, max_nonuniq, min_d, max_d, min_cov, threads=2)
    assert np.array_equal(keys, want["rare"]), "rare set differs"
    my_ptr, my_ids = c_oracle.clouds(c_oracle.unpacked_codes(batch), units, k, want["rare"])
    assert np.array_equal(csr.unit_ptr.cpu().numpy()[: units.n_units + 1], my_ptr), "local cloud sizes differ"
    assert np.array_equal(csr.ids.cpu().numpy().view(np.uint32)[: my_ids.size], my_ids), "local clouds differ"
    assert res.n_increments == want["n_increments"], (res.n_increments, want["n_increments"])
    got = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    canon = lambda e: e[np.lexsort((e[:, 3], e[:, 2], e[:, 1], e[:, 0]))]  # noqa: E731
    assert np.array_equal(canon(got), canon(want["edges"])), "edge set differs"
    assert np.array_equal(np.sort(res.selected.cpu().numpy().view(np.uint32)), want["selected"]), "unique k-mers differ"
    dist.barrier()
    if rank == 0:
        print(f"multi-gpu ok: world={world}, {rec.n_bases_total} read bases, {keys.size} rare k-mers, "
              f"{got.shape[0]} edges, {res.selected.numel()} unique k-mers, {rec.bytes_exchanged} bytes sent by rank 0")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
