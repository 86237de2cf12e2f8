"""dist.gather_eval_state, the merge behind DetectionMAP / COCODetectionEval / DetectionReport.compute(group), on CPU
tensors with gloo at world sizes 2 and 3: rank-order concatenation, padding rows never in the result, the all-empty
case, summed counts, ORed status words, and a configuration mismatch raising ValueError on every rank.

run_ranks is also the process runner of tests/test_gpu_dist_eval.py: every rank runs one function in a spawned
process with a process-group timeout, the parent collects the results with a deadline, and no child outlives the
call."""
import datetime
import os
import socket
import sys
import time
import traceback

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PG_TIMEOUT_S = 120


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _entry(rank, world, port, backend, q, fn, args):
    """One rank: join the process group, run fn(rank, world, group, *args), queue (rank, ok, result or traceback)."""
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    kw = {}
    if backend == "nccl":
        torch.cuda.set_device(rank)
        kw["device_id"] = torch.device("cuda", rank)
    dist.init_process_group(backend, rank=rank, world_size=world, timeout=datetime.timedelta(seconds=PG_TIMEOUT_S),
                            **kw)
    try:
        q.put((rank, True, fn(rank, world, dist.group.WORLD, *args)))
    except BaseException:
        q.put((rank, False, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def run_ranks(fn, world, args=(), backend="gloo", timeout_s=600):
    """fn(rank, world, group, *args) on `world` spawned ranks; returns the ranks' results in rank order.  Fails if a
    rank raised, timed out or exited non-zero; terminates and reaps every child before it returns."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=_entry, args=(r, world, port, backend, q, fn, tuple(args))) for r in range(world)]
    deadline = time.monotonic() + timeout_s
    results = {}
    try:
        for p in procs:
            p.start()
        for _ in procs:
            rank, ok, res = q.get(timeout=max(1.0, deadline - time.monotonic()))
            assert ok, f"rank {rank} failed:\n{res}"
            results[rank] = res
        for p in procs:
            p.join(timeout=max(1.0, deadline - time.monotonic()))
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
            p.join(timeout=30)
            if p.is_alive():
                p.kill()
                p.join()
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    return [results[r] for r in range(world)]


FP = (1, 3, 10, 101, 0, 0, 0, 300, 12345)


def local_state(rank, rows, width, n_counts):
    """Rank `rank`'s records: rows whose words identify (rank, row); every fifth row an unused slot (class -1)."""
    n = rows[rank]
    rec = torch.arange(n * width, dtype=torch.int32).reshape(n, width) + 1000 * (rank + 1)
    rec[:, 1] = torch.where(torch.arange(n) % 5 == 4, -1, torch.arange(n) % 3).to(torch.int32)
    counts = torch.arange(n_counts, dtype=torch.int64).reshape(-1, 2) * (rank + 1) + (1 << 40)
    status = torch.tensor([1 << rank if rank < 2 else 0], dtype=torch.int32)
    return rec, counts, 7 * (rank + 1), 2 * rank + 1, status


def merge_worker(rank, world, group, cases):
    from yolo_from_scratch_b200.dist import gather_eval_state
    out = []
    for rows, width, n_counts in cases:
        rec, counts, gt_total, images, status = local_state(rank, rows, width, n_counts)
        before = (rec.clone(), counts.clone(), status.clone())
        got = gather_eval_state(FP, rec, counts, gt_total, images, status, group)
        assert torch.equal(rec, before[0]) and torch.equal(counts, before[1]) and torch.equal(status, before[2])
        out.append((got[0].numpy(), got[1].numpy(), got[2], got[3], got[4].numpy()))
    return out


@pytest.mark.parametrize("world", [2, 3])
def test_merge_concatenates_in_rank_order(world):
    cases = [((5, 0, 13)[:world], 3, 8),      # uneven, one rank without records
             ((0, 9, 2)[:world], 8, 4),       # rank 0 empty: the others still gather
             ((0, 0, 0)[:world], 3, 6),       # every rank empty: no record exchange
             ((4, 4, 4)[:world], 3, 2)]       # equal: no padding at all
    res = run_ranks(merge_worker, world, (cases,))
    for i, (rows, width, n_counts) in enumerate(cases):
        states = [local_state(r, rows, width, n_counts) for r in range(world)]
        want_rec = np.concatenate([s[0].numpy() for s in states]).reshape(-1, width)
        want_counts = sum(s[1].numpy() for s in states)
        want_status = 0
        for s in states:
            want_status |= int(s[4])
        for r in range(world):
            rec, counts, gt_total, images, status = res[r][i]
            assert rec.dtype == np.int32 and rec.shape == (sum(rows), width)   # no padding row reaches the result
            assert np.array_equal(rec, want_rec), (r, i)
            assert counts.shape == (n_counts // 2, 2) and np.array_equal(counts, want_counts)
            assert gt_total == sum(s[2] for s in states) and images == sum(s[3] for s in states)
            assert status.dtype == np.int32 and status.tolist() == [want_status]


def mismatch_worker(rank, world, group):
    """Each case changes one configuration word on the last rank; every rank must raise, then the next case must
    still merge (no rank was left inside a collective)."""
    from yolo_from_scratch_b200.dist import gather_eval_state
    rec, counts, gt_total, images, status = local_state(rank, (3, 1, 2), 3, 4)
    last = rank == world - 1
    cases = {"nc": (FP[:1] + (FP[1] + int(last),) + FP[2:], rec, counts),
             "crc": (FP[:8] + (FP[8] ^ int(last),), rec, counts),
             "record width": (FP, torch.zeros(len(rec), 4 if last else 3, dtype=torch.int32), counts),
             "counts": (FP, rec, torch.zeros(6 if last else 4, dtype=torch.int64))}
    raised = {}
    for name, (fp, r, c) in cases.items():
        try:
            gather_eval_state(fp, r, c, gt_total, images, status, group)
            raised[name] = None
        except ValueError as e:
            raised[name] = str(e)
    after = gather_eval_state(FP, rec, counts, gt_total, images, status, group)
    return raised, after[0].shape[0]


@pytest.mark.parametrize("world", [2, 3])
def test_configuration_mismatch_raises_on_every_rank(world):
    res = run_ranks(mismatch_worker, world)
    for raised, n_after in res:
        for name, msg in raised.items():
            assert msg is not None and name in msg, (name, msg)
        assert n_after == sum((3, 1, 2)[:world])


def test_fingerprint_length_is_checked():
    from yolo_from_scratch_b200.dist import gather_eval_state
    with pytest.raises(ValueError, match="fingerprint"):
        gather_eval_state(FP[:-1], torch.zeros(0, 3, dtype=torch.int32), torch.zeros(2, dtype=torch.int64), 0, 0,
                          torch.zeros(1, dtype=torch.int32), None)
