"""bench.py's multi-rank end-to-end region on CPU (gloo, 2 ranks, a fake scan): the number is the slowest rank's, a
parity mismatch on one rank is seen by all, and a failure on ONE rank drops the number everywhere without hanging."""
import os
import socket
import sys
import time

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, scenario, q):
    sys.path.insert(0, ROOT)
    import bench
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    want = np.arange(5, dtype=np.uint64)

    def scan():
        time.sleep(0.05 if rank == 1 else 0.01)
        if scenario == "raise" and rank == 1:
            raise RuntimeError("boom")
        return want + (1 if scenario == "mismatch" and rank == 0 else 0)

    fn = None if (scenario == "setup_failed" and rank == 0) else scan
    res = bench.e2e_all_ranks(fn, want.tobytes(), 3, world, rank, torch, dist, "cpu", dist.barrier)
    q.put((rank, res))
    dist.barrier()
    dist.destroy_process_group()


def _run(scenario):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, scenario, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def test_slowest_rank_sets_the_time():
    res = _run("ok")
    assert res[0] is not None and res[1] is not None
    assert abs(res[0][0] - res[1][0]) < 1e-9 and res[0][0] >= 0.045  # rank 1 sleeps 50 ms per step
    assert res[0][1] == 5 and res[0][2] and res[1][2]


def test_mismatch_on_one_rank_is_seen_by_all():
    res = _run("mismatch")
    assert res[0][2] is False and res[1][2] is False


def test_failure_on_one_rank_drops_the_number_without_hanging():
    assert _run("raise") == {0: None, 1: None}
    assert _run("setup_failed") == {0: None, 1: None}


def test_dump_records_exact_and_bounded(tmp_path):
    """--dump-outputs: every field as exact float64; above the byte budget a fixed-seed sample of rows, the same one on
    every run, within the budget."""
    sys.path.insert(0, ROOT)
    import bench
    from grab_b200 import MATCH_DTYPE
    r = np.zeros(1000, dtype=MATCH_DTYPE)
    r["start"] = np.arange(1000, dtype=np.uint64) * np.uint64(1 << 40) + np.uint64(7)
    r["file_id"] = np.arange(1000) * 3
    r["match_len"] = 15
    bench.dump_records(r, str(tmp_path / "all"), "", 1 << 20)
    for f in ("start", "file_id", "match_len"):
        got = np.load(tmp_path / "all" / (f + ".npy"))
        assert got.dtype == np.float64 and np.array_equal(got.astype(np.uint64), r[f])
    assert not (tmp_path / "all" / "sample_rows.npy").exists()
    for d in ("s1", "s2"):
        bench.dump_records(r, str(tmp_path / d), "", 3200)
    rows = np.load(tmp_path / "s1" / "sample_rows.npy")
    assert len(rows) == 100 and np.array_equal(rows, np.load(tmp_path / "s2" / "sample_rows.npy"))
    assert np.array_equal(np.load(tmp_path / "s1" / "start.npy").astype(np.uint64), r["start"][rows.astype(np.int64)])
    assert sum(os.path.getsize(tmp_path / "s1" / f) - 128 for f in os.listdir(tmp_path / "s1")) <= 3200
