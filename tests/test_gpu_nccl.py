"""The one collective of the path (SURVEY 8(e)): the end-of-run all-gather of the per-episode records over NCCL, two
ranks on two GPUs of one box.  Skipped on a one-GPU box (the gloo twin of this test, tests/test_sharding.py, runs on CPU)."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOTAL = 1001   # odd: the blocks differ in size by one


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, ws, port, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(ws), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    try:
        from deepgroebner_b200 import sharding
        from deepgroebner_b200.buchberger import BuchbergerEngine
        eng = BuchbergerEngine("3-20-10-weighted", num_envs=256, device="cuda:%d" % rank)
        out = {}
        for strategy in ("degree", "random"):
            rec = sharding.run_sharded(eng, strategy, TOTAL, seed_base=20, compute_gb=True, selection_seed=5)
            out[strategy] = rec.tobytes()
        q.put((rank, out))
    finally:
        dist.destroy_process_group()


def test_gather_records_over_nccl_two_ranks():
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from oracle import oracle as O
    from test_gpu_parity import assert_records_equal, reference_records
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    dt = np.dtype(O.Oracle.RECORD_DTYPE)
    for strategy in ("degree", "random"):
        want = reference_records("3-20-10-weighted", strategy, TOTAL, seed0=20, sel_seed0=5)
        for rank in (0, 1):
            rec = np.frombuffer(got[rank][strategy], dtype=dt)
            assert rec.shape == (TOTAL,)
            assert_records_equal(rec, want, "%s, rank %d" % (strategy, rank))
