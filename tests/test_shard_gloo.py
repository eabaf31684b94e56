"""world_size-2 gloo test (CPU) of the N>1 host logic: contiguous spectrum shards, per-rank scoring, gather on rank 0,
result identical (order and rebased spectrum indices) to a single-process run. The per-rank scorer here is the oracle —
the sharding logic is independent of what scores a shard."""
import os
import socket
import sys

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, tmp):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from sage_b200 import synth
    from sage_b200.shard import score_sharded
    from helpers import oracle_db_from_peptides
    from oracle import oracle as O
    pep = synth.make_peptides(4000, seed=31)
    spectra = synth.make_spectra(pep, 101, seed=32)  # odd count: uneven shards
    odb = oracle_db_from_peptides(pep)
    cfg = O.ScorerConfig(precursor_tol=(O.PPM, -20, 20), fragment_tol=(O.PPM, -20, 20), report_psms=2)

    def score_fn(b):
        f, c, _, _ = odb.score_batch(cfg, b.as_dict(), nthreads=1)
        return f, c
    res = score_sharded(score_fn, spectra, 2, rank, world, dist=dist)
    if rank == 0:
        f, c = res
        np.save(os.path.join(tmp, "f.npy"), f)
        np.save(os.path.join(tmp, "c.npy"), c)
        f1, c1 = score_fn(spectra)
        np.save(os.path.join(tmp, "f1.npy"), f1)
        np.save(os.path.join(tmp, "c1.npy"), c1)
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:   # a port the OS just handed out: on a shared host a fixed or pid-derived one may be taken
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_sharded_equals_single(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    f, c = np.load(tmp_path / "f.npy"), np.load(tmp_path / "c.npy")
    f1, c1 = np.load(tmp_path / "f1.npy"), np.load(tmp_path / "c1.npy")
    assert np.array_equal(c, c1)
    sel = (np.arange(len(f)) % 2) < np.repeat(c, 2)
    assert f[sel].tobytes() == f1[sel].tobytes()


def test_shard_ranges_cover():
    from sage_b200.shard import shard_range
    for n in (0, 1, 7, 50_000, 200_000):
        for w in (1, 2, 4, 8):
            r = [shard_range(n, w, k) for k in range(w)]
            assert r[0][0] == 0 and r[-1][1] == n and all(r[i][1] == r[i + 1][0] for i in range(w - 1))
