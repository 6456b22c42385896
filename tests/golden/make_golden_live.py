"""Record the reference's outputs on the inputs of tests/test_oracle_vs_live_reference.py and
tests/test_drop_in_reference.py, by RUNNING THE REFERENCE ITSELF on CPU (imported in place, read-only, comet_ml
stubbed as in make_golden.py).  Output: tests/golden/reference_golden_live.npz, committed.  An output of more than
4096 elements is stored as its shape and a fixed, seeded sample of its elements.

    python tests/golden/make_golden_live.py <the reference checkout's src directory>
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import make_golden as G  # noqa: E402
import make_golden_balancing as GB  # noqa: E402
import make_golden_mase as GM  # noqa: E402
import test_drop_in_reference as D  # noqa: E402
import test_oracle_vs_live_reference as T  # noqa: E402
from oracle import al_oracle as O  # noqa: E402

SAMPLE = 4096


def put(gold, key, x, seed):
    x = np.asarray(x)
    if x.size > SAMPLE:
        at = np.sort(np.random.default_rng(seed).choice(x.size, SAMPLE, replace=False))
        gold[key + "_at"], gold[key + "_shape"], x = at, np.array(x.shape), x.ravel()[at]
    gold[key] = x


def main(src):
    G.REF = src
    get_strategy, Exp = G._import_reference()
    gold = {}
    for seed in range(3):
        ev, lab, lb, logits = T.margin_inputs(seed)
        s = G.make_strategy(get_strategy, Exp, "MarginSampler", logits, torch.zeros(len(lb), 4), ev, lab, 64)
        idx, cost = s.query(50.0)
        gold[f"margin{seed}_idx"], gold[f"margin{seed}_cost"] = np.array(idx, dtype=np.int64), np.array(cost)

        feat, ind = T.pairwise_inputs(seed)
        cs = get_strategy("CoresetSampler")
        obj = cs.__new__(cs)
        d2 = obj.get_pairwise_l2_dist(feat)
        put(gold, f"pairwise{seed}_d2", d2.numpy(), seed)
        gold[f"pairwise{seed}_greedy"] = np.array(obj.coreset(d2, ind, 30, randomize=False), dtype=np.int64)
        np.random.seed(seed)
        gold[f"pairwise{seed}_d2sample"] = np.array(obj.coreset(d2, ind, 30, randomize=True), dtype=np.int64)
        none = np.zeros(len(ind), dtype=bool)
        gold[f"pairwise{seed}_cold"] = np.array(obj.coreset(d2, none, 4, randomize=False), dtype=np.int64)

        ev, lab, lb, emb, w, b, bs, budget = T.mase_inputs(seed)
        avail = O.available_query_idxs(lb, ev, shuffle=False)
        for name, key in (("MASESampler", "mase_picks"), ("BASESampler", "base_picks")):
            s = GM.make_strategy(get_strategy, Exp, name, emb, w, b, ev, lab, bs)
            with GM._cuda_is_identity():
                gold[f"mase{seed}_{key}"] = np.array(s.query(float(budget))[0], dtype=np.int64)
                mm, pc, pred, _ = s.compute_margins(avail)
        put(gold, f"mase{seed}_mm", mm.numpy(), seed)
        put(gold, f"mase{seed}_pc", pc.numpy(), seed)
        put(gold, f"mase{seed}_pred", pred.numpy(), seed)

        ev, lab, lb, emb, ys, c, budget = T.balancing_inputs(seed)
        idx, cost = GB.run_reference(get_strategy, Exp, emb, ys, c, ev, lab, 64, budget, seed)
        gold[f"balancing{seed}_idx"], gold[f"balancing{seed}_cost"] = np.array(idx, dtype=np.int64), np.array(cost)

    for seed in range(2):
        lg, h, bs = T.gradient_inputs(seed)
        s = G.make_strategy(get_strategy, Exp, "BADGESampler", lg, h, [], [], bs)
        for pooled in (False, True):
            put(gold, f"grad{seed}_{int(pooled)}",
                s.get_gradient_embeddings(list(range(len(lg))), use_adaptive_pool=pooled).numpy(), seed)

    for case, (name, kw, budget) in enumerate(D.CASES):
        logits, emb, ev, lab = D.inputs()
        s = D._build(get_strategy(name), Exp(), logits, emb, ev, lab, 64, **kw)
        np.random.seed(9)
        idx, cost = s.query(budget)
        gold[f"dropin{case}_picks"], gold[f"dropin{case}_cost"] = np.array([int(i) for i in idx]), np.array(cost)

    path = os.path.join(HERE, "reference_golden_live.npz")
    np.savez_compressed(path, **gold)
    print("wrote", len(gold), "arrays ->", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
