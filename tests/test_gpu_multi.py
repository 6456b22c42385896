"""Multi-GPU (one process per GPU, NCCL + peer-memory windows): results must equal the single-GPU /
reference results for every world size.  Needs >= 2 GPUs (skipped otherwise; on a machine with two, run
`python -m pytest tests/test_gpu_multi.py -m gpu`)."""
import os
import socket
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _worker(rank, world, port, gold_path, out_path):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from helpers import load_gold, make_strategy
    from active_learning_b200.engine import Engine
    from active_learning_b200.sharding import ShardGroup
    gold = load_gold(gold_path)
    n, ev, lab = int(gold["e2e_n"]), gold["e2e_eval_idxs"], gold["e2e_labeled"]
    eng = Engine(rank).comm_init()
    group = ShardGroup()
    res = {}

    def run(name, key, logits, emb, labeled, budget, seed, **kw):
        s = make_strategy(name, logits, emb, ev, labeled, 64, engine=eng, **kw)
        s._shard_group = group
        np.random.seed(seed)
        idx, cost = s.query(budget)
        res[key] = [int(i) for i in idx]
        assert cost == len(idx)

    lg = torch.from_numpy(gold["e2e_logits"])
    for etag in ("int", "f32"):
        emb = torch.from_numpy(gold[f"e2e_emb_{etag}"])
        run("CoresetSampler", f"e2e_CoresetSampler_all_{etag}", lg, emb, lab, 50.0, 21)
        run("CoresetSampler", f"e2e_CoresetSampler_sub_{etag}", lg, emb, lab, 50.0, 21, subset_labeled=60, subset_unlabeled=300)
        run("BADGESampler", f"e2e_BADGESampler_sub_{etag}", lg, emb, lab, 50.0, 21, subset_labeled=60, subset_unlabeled=300)
        run("PartitionedCoresetSampler", f"e2e_PartitionedCoresetSampler_sub_{etag}", lg, emb, lab, 50.0, 21,
            partitions=3, subset_labeled=60, subset_unlabeled=300)
        run("PartitionedBADGESampler", f"e2e_PartitionedBADGESampler_sub_{etag}", lg, emb, lab, 50.0, 21,
            partitions=3, subset_labeled=60, subset_unlabeled=300)
    for tag in ("f32_c10", "f32_c1000"):
        run("MarginSampler", f"margin_{tag}_picks", torch.from_numpy(gold[f"margin_{tag}_logits"]), torch.zeros(n, 4),
            lab, 60.0, 7)
    # nothing labeled: first centre by minimax / np.random.choice, compared with the single-GPU engine path
    emb = torch.from_numpy(gold["e2e_emb_int"])
    for name in ("CoresetSampler", "BADGESampler"):
        run(name, f"cold_{name}_multi", lg, emb, [], 12.0, 5)
        s = make_strategy(name, lg, emb, ev, [], 64, engine=eng)
        np.random.seed(5)
        res[f"cold_{name}_single"] = [int(i) for i in s.query(12.0)[0]]
    # MASE (rows sharded, one top-B exchange) and BASE (margins sharded + gathered, class loop replicated)
    from helpers import HeadNet
    mg = dict(np.load(os.path.join(ROOT, "tests", "golden", "reference_golden_mase.npz")))
    for tag in ("a", "b"):
        for name, key in (("MASESampler", "mase"), ("BASESampler", "base")):
            net = HeadNet(torch.from_numpy(mg[f"{tag}_emb"]), torch.from_numpy(mg[f"{tag}_weight"]), torch.from_numpy(mg[f"{tag}_bias"]))
            s = make_strategy(name, None, None, mg[f"{tag}_eval"], mg[f"{tag}_labeled"], int(mg[f"{tag}_bs"]), engine=eng, net=net)
            s._shard_group = group
            res[f"mgold_{tag}_{key}_picks"] = [int(i) for i in s.query(float(mg[f"{tag}_budget"]))[0]]
    ranks_agree = [None] * world
    dist.all_gather_object(ranks_agree, res)
    assert all(r == res for r in ranks_agree)
    if rank == 0:
        np.save(out_path, np.array([res], dtype=object), allow_pickle=True)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_equal_reference(gold):
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = os.path.join(tempfile.mkdtemp(), "res.npy")
    mp.spawn(_worker, args=(2, port, os.path.join(ROOT, "tests", "golden", "reference_golden.npz"), out),
             nprocs=2, join=True)
    res = np.load(out, allow_pickle=True)[0]
    mg = dict(np.load(os.path.join(ROOT, "tests", "golden", "reference_golden_mase.npz")))
    for key, got in res.items():
        if key.startswith("cold_"):
            continue
        if key.startswith("mgold_"):
            assert got == mg[key[len("mgold_"):]].tolist(), key
            continue
        assert got == gold[key].tolist(), key
    for name in ("CoresetSampler", "BADGESampler"):
        assert res[f"cold_{name}_multi"] == res[f"cold_{name}_single"], name
