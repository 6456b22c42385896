"""Generate the golden vectors under tests/golden/ by RUNNING THE REFERENCE ITSELF.

Only runs in the build container (needs /root/reference).  The reference is imported in place,
read-only, with a stub for the one missing dependency (comet_ml).  Outputs are small .npz
files committed next to this script; tests replay them against oracle/ (CPU) and against the
CUDA path (GPU).  Nothing at test/bench time reads /root/reference.

    python tests/golden/make_golden.py
"""
import os
import sys
import tempfile
import types

import numpy as np
import torch
import torch.nn as nn

REF = "/root/reference/src"
OUT = os.path.dirname(os.path.abspath(__file__))


# --- import the reference -----------------------------------------------------------------
def _import_reference():
    stub = types.ModuleType("comet_ml")

    class _Exp:
        url = "."

        def __init__(self, *a, **k):
            pass

        def get_key(self):
            return "golden"

        def __getattr__(self, name):
            return lambda *a, **k: None

    stub.Experiment = _Exp
    stub.ExistingExperiment = _Exp
    sys.modules["comet_ml"] = stub
    sys.path.insert(0, REF)
    from query_strategies.get_strategy import get_strategy  # noqa
    return get_strategy, _Exp


class IndexDataset(torch.utils.data.Dataset):
    """al_set stand-in: x is the sample's own index, so a lookup 'network' can return any
    logits/embedding we choose for it (custom_imagenet.py:24-26 yields (x, y, index))."""

    def __init__(self, n, num_classes):
        self.n, self.num_classes = n, num_classes
        self.targets = [0] * n

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        return torch.tensor(float(i)), 0, i


class LookupNet(nn.Module):
    """net(x) -> logits[x]; net(x, return_features=...) -> (logits[x], emb[x])
    (models/resnet_simclr.py:29-41)."""

    def __init__(self, logits, emb):
        super().__init__()
        self.register_buffer("logits", logits)
        self.register_buffer("emb", emb)
        self.dummy = nn.Parameter(torch.zeros(1))

    def forward(self, x, return_features=False, specify_input_layer=None):
        i = x.long()
        if return_features:
            return self.logits[i], self.emb[i]
        return self.logits[i]


def make_strategy(get_strategy, Exp, name, logits, emb, eval_idxs, labeled, batch_size, **kw):
    n, c = logits.shape
    ds = IndexDataset(n, c)
    net = LookupNet(logits, emb)
    tmp = tempfile.mkdtemp(prefix="golden_")
    args = dict(early_stop_patience=0, n_epoch=1, world_size=1, model="SSLResNet18",
                freeze_feature=True, ckpt_path=tmp, exp_name="g", subset_labeled=None,
                subset_unlabeled=None, partitions=1)
    args.update(kw)
    train_args = {"loader_te_args": {"batch_size": batch_size, "num_workers": 0}}
    s = get_strategy(name)(ds, ds, net, train_args, np.array(eval_idxs), Exp(), None, **args)
    s.feature_net = s.net  # what init_network_weights does (strategy.py:198)
    if len(labeled):
        s.update(np.array(labeled), len(labeled))
    return s


def dyadic_logits(rng, n, c):
    """Multiples of 1/4 in [-6, 6]: plenty of exact ties for the tie-break rules."""
    return torch.from_numpy(rng.integers(-24, 25, size=(n, c)).astype(np.float32) / 4.0)


def main():
    get_strategy, Exp = _import_reference()
    torch.manual_seed(0)
    rng = np.random.default_rng(1234)
    gold = {}

    # ---------------------------------------------------------------- pool bookkeeping
    n = 700
    eval_idxs = rng.choice(n, size=40, replace=False)
    rest = np.setdiff1d(np.arange(n), eval_idxs)
    labeled = rng.choice(rest, size=90, replace=False)

    # ---------------------------------------------------------------- Margin (A1)
    for tag, c, mk in (("f32_c10", 10, None), ("f32_c1000", 1000, None), ("dyadic_c10", 10, 1)):
        logits = dyadic_logits(rng, n, c) if mk else torch.randn(n, c) * 3.0
        emb = torch.zeros(n, 4)
        s = make_strategy(get_strategy, Exp, "MarginSampler", logits, emb, eval_idxs, labeled, 128)
        np.random.seed(7)
        idx, cost = s.query(60.0)
        gold[f"margin_{tag}_logits"] = logits.numpy()
        gold[f"margin_{tag}_picks"] = np.array(idx, dtype=np.int64)
        assert cost == 60
    # 2.8 MB: tests/helpers.py regenerates these logits from the seed and checks them against this sample
    gold["margin_f32_c1000_logits_sample"] = gold.pop("margin_f32_c1000_logits")[::7, ::13]

    # ---------------------------------------------------------------- Confidence (A2)
    # As shipped the reference raises (confidence_sampler.py:41).  Record that, then record the
    # intended behaviour: the same source with line 41 dropped, exec'd in the module's namespace.
    import query_strategies.confidence_sampler as cs
    logits = torch.randn(n, 10) * 3.0
    s = make_strategy(get_strategy, Exp, "ConfidenceSampler", logits, torch.zeros(n, 4),
                      eval_idxs, labeled, 128)
    np.random.seed(7)
    try:
        s.query(60.0)
        gold["confidence_raises"] = np.array(0)
    except IndexError:
        gold["confidence_raises"] = np.array(1)
    src = open(cs.__file__).read().splitlines()
    assert "confidence = confidence[idxs_for_query]" in src[40], src[40]
    del src[40]
    ns = dict(vars(cs))
    exec(compile("\n".join(src), "confidence_sampler_minus_line41", "exec"), ns)
    s.__class__ = ns["ConfidenceSampler"]
    for tag, lg in (("f32", logits), ("dyadic", dyadic_logits(rng, n, 10))):
        s.net = LookupNet(lg, torch.zeros(n, 4))
        np.random.seed(7)
        idx, cost = s.query(60.0)
        gold[f"confidence_{tag}_logits"] = lg.numpy()
        gold[f"confidence_{tag}_picks"] = np.array(idx, dtype=np.int64)

    # ---------------------------------------------------------------- pairwise + coreset (A7-A9)
    cs_obj = get_strategy("CoresetSampler").__new__(get_strategy("CoresetSampler"))
    m, d, l0, b = 320, 64, 45, 40
    feat_int = torch.from_numpy(rng.integers(-1, 2, size=(m, d)).astype(np.float32))
    feat_f32 = torch.relu(torch.randn(m, d))
    ind = np.zeros(m, dtype=bool)
    ind[rng.choice(m, size=l0, replace=False)] = True
    gold["cs_indicator"] = ind
    for tag, feat in (("int", feat_int), ("f32", feat_f32)):
        d2 = cs_obj.get_pairwise_l2_dist(feat)
        gold[f"cs_{tag}_feat"] = feat.numpy()
        gold[f"cs_{tag}_d2"] = d2.numpy()
        gold[f"cs_{tag}_greedy"] = np.array(cs_obj.coreset(d2, ind, b, randomize=False))
        np.random.seed(11)
        gold[f"cs_{tag}_d2sample"] = np.array(cs_obj.coreset(d2, ind, b, randomize=True))
        # nothing labeled: minimax first centre / uniform first draw (coreset_sampler.py:97-100)
        none = np.zeros(m, dtype=bool)
        gold[f"cs_{tag}_greedy_cold"] = np.array(cs_obj.coreset(d2, none, 6, randomize=False))
        np.random.seed(12)
        gold[f"cs_{tag}_d2sample_cold"] = np.array(cs_obj.coreset(d2, none, 6, randomize=True))
    # duplicates of labeled rows: the sum(prob)==0 -> NaN -> += 1e-5 retry branch (:87-90)
    feat_dup = feat_int[:8].repeat(6, 1)
    ind_dup = np.zeros(48, dtype=bool)
    ind_dup[:8] = True
    d2 = cs_obj.get_pairwise_l2_dist(feat_dup)
    np.random.seed(13)
    gold["cs_dup_feat"] = feat_dup.numpy()
    gold["cs_dup_indicator"] = ind_dup
    gold["cs_dup_d2sample"] = np.array(cs_obj.coreset(d2, ind_dup, 5, randomize=True))

    # ---------------------------------------------------------------- gradient embeddings (A11)
    ng, cg, dg, bs = 53, 10, 16, 16   # 53 % 16 = 5: short last batch
    lg = torch.randn(ng, cg) * 3.0
    hg = torch.relu(torch.randn(ng, dg))
    s = make_strategy(get_strategy, Exp, "BADGESampler", lg, hg, [], [], bs)
    gold["ge_logits"], gold["ge_emb"] = lg.numpy(), hg.numpy()
    gold["ge_full"] = s.get_gradient_embeddings(list(range(ng))).numpy()
    gold["ge_pooled"] = s.get_gradient_embeddings(list(range(ng)), use_adaptive_pool=True).numpy()
    ng2, cg2, dg2 = 9, 40, 96         # C > 16: pool to (16, 32)
    lg2 = torch.randn(ng2, cg2) * 3.0
    hg2 = torch.relu(torch.randn(ng2, dg2))
    s = make_strategy(get_strategy, Exp, "BADGESampler", lg2, hg2, [], [], 4)
    gold["ge2_logits"], gold["ge2_emb"] = lg2.numpy(), hg2.numpy()
    gold["ge2_pooled"] = s.get_gradient_embeddings(list(range(ng2)), use_adaptive_pool=True).numpy()

    # ---------------------------------------------------------------- end-to-end query() (A10, A12-A14)
    c_e, d_e = 10, 32
    logits_e = torch.randn(n, c_e) * 3.0
    emb_int = torch.from_numpy(rng.integers(-1, 2, size=(n, d_e)).astype(np.float32))
    emb_f32 = torch.relu(torch.randn(n, d_e))
    gold["e2e_logits"] = logits_e.numpy()
    gold["e2e_emb_int"] = emb_int.numpy()
    gold["e2e_emb_f32"] = emb_f32.numpy()
    gold["e2e_eval_idxs"] = eval_idxs
    gold["e2e_labeled"] = labeled
    gold["e2e_n"] = np.array(n)
    for name, kw in (("CoresetSampler", {}),
                     ("CoresetSampler", dict(subset_labeled=60, subset_unlabeled=300)),
                     ("PartitionedCoresetSampler", dict(partitions=3, subset_labeled=60,
                                                        subset_unlabeled=300)),
                     ("BADGESampler", dict(subset_labeled=60, subset_unlabeled=300)),
                     ("PartitionedBADGESampler", dict(partitions=3, subset_labeled=60,
                                                      subset_unlabeled=300))):
        for etag, emb in (("int", emb_int), ("f32", emb_f32)):
            s = make_strategy(get_strategy, Exp, name, logits_e, emb, eval_idxs, labeled, 64, **kw)
            np.random.seed(21)
            idx, cost = s.query(50.0)
            key = f"e2e_{name}_{'sub' if kw.get('subset_labeled') else 'all'}_{etag}"
            gold[key] = np.array([int(i) for i in idx], dtype=np.int64)
            assert cost == 50, (name, cost)

    # ---------------------------------------------------------------- np.random.choice == cdf search
    p = rng.random(1000).astype(np.float32)
    p[rng.choice(1000, 300, replace=False)] = 0
    p = p / np.sum(p)
    np.random.seed(5)
    draws = [int(np.random.choice(len(p), p=p)) for _ in range(64)]
    np.random.seed(5)
    us = np.random.random_sample(64)
    gold["choice_p"], gold["choice_draws"], gold["choice_uniforms"] = p, np.array(draws), us

    np.savez_compressed(os.path.join(OUT, "reference_golden.npz"), **gold)
    print("wrote", len(gold), "arrays ->", os.path.join(OUT, "reference_golden.npz"),
          os.path.getsize(os.path.join(OUT, "reference_golden.npz")), "bytes")


if __name__ == "__main__":
    main()
