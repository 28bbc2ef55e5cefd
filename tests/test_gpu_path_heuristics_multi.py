"""Two-rank NCCL run of the collective Katz / PPR calls (plnlp_b200/paths.py) on a row-partitioned graph: every
score, id and rank bit-identical to one GPU, and a call whose method parameters differ between the ranks raising
ValueError on every rank.  Skipped below 2 GPUs."""
import pytest
import torch
import torch.multiprocessing as mp

from tests.test_gpu_path_heuristics import _free_port, check, worker

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_collective_two_ranks_nccl():
    ret = mp.Manager().dict()
    mp.spawn(worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    check(ret, 2)
