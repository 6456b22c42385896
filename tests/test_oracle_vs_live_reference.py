"""The oracle against the reference on fresh random inputs (beyond the fixtures of make_golden*.py).

Inputs are drawn here from their seeds.  tests/golden/make_golden_live.py ran the reference (imported in place,
comet_ml stubbed) on the same inputs and stored what it returned in reference_golden_live.npz; an output of more
than 4096 elements is stored as its shape and a fixed, seeded sample of its elements.  Every comparison is exact:
the oracle runs the same torch-CPU / NumPy arithmetic in the same order."""
import os

import numpy as np
import pytest
import torch

from oracle import al_oracle as O

LIVE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden_live.npz")


@pytest.fixture(scope="module")
def ref():
    return dict(np.load(LIVE))


def same(x, ref, key):
    """x equals the reference's output `key` (or, where only a sample was stored, its shape and sampled elements)."""
    x = np.asarray(x)
    if key + "_at" in ref:
        return x.shape == tuple(ref[key + "_shape"]) and np.array_equal(x.ravel()[ref[key + "_at"]], ref[key])
    return np.array_equal(x, ref[key])


def pool(rng, n, n_eval, n_lab):
    ev = rng.choice(n, size=n_eval, replace=False)
    rest = np.setdiff1d(np.arange(n), ev)
    lab = rng.choice(rest, size=n_lab, replace=False)
    lb = np.zeros(n, dtype=bool)
    lb[lab] = True
    return ev, lab, lb


def margin_inputs(seed):
    rng = np.random.default_rng(seed)
    torch.manual_seed(seed)
    n, c = 300 + 17 * seed, (10, 100, 37)[seed]
    ev, lab, lb = pool(rng, n, 20, 40)
    return ev, lab, lb, torch.randn(n, c) * 3


def pairwise_inputs(seed):
    rng = np.random.default_rng(10 + seed)
    torch.manual_seed(10 + seed)
    m, d = 200 + 31 * seed, (16, 48, 7)[seed]
    feat = torch.relu(torch.randn(m, d))
    ind = np.zeros(m, dtype=bool)
    ind[rng.choice(m, size=25, replace=False)] = True
    return feat, ind


def gradient_inputs(seed):
    torch.manual_seed(20 + seed)
    n, c, d, bs = (45, 70)[seed], (10, 24)[seed], (12, 40)[seed], (16, 32)[seed]
    lg, h = torch.randn(n, c) * 3, torch.relu(torch.randn(n, d))
    return lg, h, bs


def mase_inputs(seed):
    rng = np.random.default_rng(30 + seed)
    torch.manual_seed(30 + seed)
    n, m, c, bs, budget = 260, (8, 24, 16)[seed], (5, 12, 40)[seed], 64, 36
    ev, lab, lb = pool(rng, n, 15, 30)
    # + rand: no all-zero rows -> no exactly equal margins (the reference's torch.sort is not stable on ties)
    emb, w, b = torch.relu(torch.randn(n, m)) + 0.05 * torch.rand(n, m), torch.randn(c, m) * 0.5, torch.randn(c) * 0.1
    return ev, lab, lb, emb, w, b, bs, budget


def balancing_inputs(seed):
    rng = np.random.default_rng(40 + seed)
    torch.manual_seed(40 + seed)
    n, m, c, budget = 240, 10, (4, 6, 3)[seed], (30, 24, 40)[seed]
    probs = np.array([0.5, 0.25, 0.15, 0.05, 0.03, 0.02][:c])
    ys = rng.choice(c, size=n, p=probs / probs.sum())
    emb = torch.relu(torch.randn(c, m)[torch.from_numpy(ys)] * 2 + torch.randn(n, m))
    ev, lab, lb = pool(rng, n, 12, (40, 25, 60)[seed])
    return ev, lab, lb, emb, ys, c, budget


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_margin_query(ref, seed):
    ev, lab, lb, logits = margin_inputs(seed)
    avail = O.available_query_idxs(lb, ev, shuffle=False)
    mine, mcost = O.uncertainty_query(logits[avail], avail, 50.0, O.MODE_MARGIN)
    assert mine == ref[f"margin{seed}_idx"].tolist() and mcost == ref[f"margin{seed}_cost"]


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_pairwise_and_both_coreset_modes(ref, seed):
    feat, ind = pairwise_inputs(seed)
    d2 = O.pairwise_l2_dist(feat)
    assert same(d2.numpy(), ref, f"pairwise{seed}_d2")
    greedy, want = ref[f"pairwise{seed}_greedy"].tolist(), ref[f"pairwise{seed}_d2sample"].tolist()
    assert O.coreset(d2, ind, 30, randomize=False) == greedy
    assert O.coreset_streaming(feat, ind, 30) == greedy
    np.random.seed(seed)
    assert O.coreset(d2, ind, 30, randomize=True) == want
    np.random.seed(seed)                                      # the O(N)-memory form with NumPy-exact sampling arithmetic
    assert O.coreset_streaming(feat, ind, 30, randomize=True) == want
    none = np.zeros(len(ind), dtype=bool)                     # cold start: minimax centre / uniform draw
    assert O.coreset(d2, none, 4, randomize=False) == ref[f"pairwise{seed}_cold"].tolist()


@pytest.mark.parametrize("seed", [0, 1])
def test_gradient_embeddings(ref, seed):
    lg, h, bs = gradient_inputs(seed)
    for pooled in (False, True):
        assert same(O.gradient_embeddings(lg, h, bs, use_adaptive_pool=pooled).numpy(), ref, f"grad{seed}_{int(pooled)}")


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_mase_and_base(ref, seed):
    ev, lab, lb, emb, w, b, bs, budget = mase_inputs(seed)
    avail = O.available_query_idxs(lb, ev, shuffle=False)
    omm, opc, opred = O.mase_margins(emb[avail], w, b, bs)
    k = f"mase{seed}"
    assert same(omm.numpy(), ref, f"{k}_mm") and same(opc.numpy(), ref, f"{k}_pc") and same(opred.numpy(), ref, f"{k}_pred")
    assert O.mase_query(omm, avail, float(budget))[0] == ref[f"{k}_mase_picks"].tolist()
    assert avail[O.base_select(omm, opc, opred, budget, w.shape[0])].tolist() == ref[f"{k}_base_picks"].tolist()


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_balancing(ref, seed):
    ev, lab, lb, emb, ys, c, budget = balancing_inputs(seed)
    avail = ~lb
    avail[ev] = False
    np.random.seed(seed)
    mine, mcost = O.balancing_query(emb, torch.from_numpy(ys), avail, lb, float(budget), c)
    assert mine == ref[f"balancing{seed}_idx"].tolist() and mcost == ref[f"balancing{seed}_cost"]
