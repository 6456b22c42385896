"""INTEGRATION.md's three-line patch, executed: `make_drop_in` binds the accelerated query() implementations onto the
Strategy base class it is given -- here the package's own query-path Strategy, which keeps the reference's
constructor contract and bookkeeping -- and the resulting classes' query(), arithmetic by the CPU oracle engine as
everywhere in the CPU tier, must return exactly what the reference's own samplers returned on the same pool, labels
and RNG seed (recorded by tests/golden/make_golden_live.py in reference_golden_live.npz)."""
import os
import tempfile

import numpy as np
import pytest
import torch

from active_learning_b200.integration import make_drop_in
from active_learning_b200.query_strategies.strategy import Strategy

LIVE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden_live.npz")


@pytest.fixture(scope="module")
def ref():
    return dict(np.load(LIVE))


def _build(cls, exp, logits, emb, ev, lab, bs, **kw):
    from helpers import IndexDataset, LookupNet, OracleEngine
    n, c = logits.shape
    ds = IndexDataset(n, c)
    net = LookupNet(logits, emb)
    args = dict(early_stop_patience=0, n_epoch=1, world_size=1, model="SSLResNet18", freeze_feature=True,
                ckpt_path=tempfile.mkdtemp(prefix="dropin_"), exp_name="d", subset_labeled=None, subset_unlabeled=None,
                partitions=1)
    args.update(kw)
    s = cls(ds, ds, net, {"loader_te_args": {"batch_size": bs, "num_workers": 0}}, np.array(ev), exp, None, **args)
    s.feature_net = s.net            # what the reference's init_network_weights does (strategy.py:198)
    if hasattr(s, "set_engine"):
        s.set_engine(OracleEngine())
    if len(lab):
        s.update(np.array(lab), len(lab))
    return s


CASES = [
    ("MarginSampler", {}, 60.0),
    ("CoresetSampler", {}, 40.0),
    ("CoresetSampler", dict(subset_labeled=50, subset_unlabeled=200), 40.0),
    ("BADGESampler", dict(subset_labeled=50, subset_unlabeled=200), 40.0),
    ("PartitionedCoresetSampler", dict(partitions=3, subset_labeled=50, subset_unlabeled=240), 40.0),
    ("PartitionedBADGESampler", dict(partitions=3, subset_labeled=50, subset_unlabeled=240), 40.0),
]


def inputs():
    rng = np.random.default_rng(5)
    torch.manual_seed(5)
    n, c, d = 420, 10, 32
    ev = rng.choice(n, size=30, replace=False)
    rest = np.setdiff1d(np.arange(n), ev)
    lab = rng.choice(rest, size=70, replace=False)
    logits = torch.randn(n, c) * 3
    emb = torch.from_numpy(rng.integers(-2, 3, size=(n, d)).astype(np.float32))     # exact arithmetic: order-free sums
    return logits, emb, ev, lab


@pytest.mark.parametrize("name,kw,budget", CASES)
def test_drop_in_classes_on_the_reference_strategy_return_the_reference_picks(ref, name, kw, budget):
    from helpers import FakeExperiment
    case = CASES.index((name, kw, budget))
    logits, emb, ev, lab = inputs()
    accel = make_drop_in(Strategy)
    mine = _build(accel[name], FakeExperiment(), logits, emb, ev, lab, 64, **kw)
    # the accelerated class IS a Strategy of the base it was bound to: training, checkpointing, update() are the base's
    assert isinstance(mine, Strategy) and Strategy in type(mine).__mro__
    assert type(mine).train is Strategy.train and type(mine).update is Strategy.update
    np.random.seed(9)
    got, got_cost = mine.query(budget)
    assert [int(i) for i in got] == ref[f"dropin{case}_picks"].tolist() and got_cost == ref[f"dropin{case}_cost"]
    # the consumer of query()'s return: update() accepts it (asserts not-yet-labeled, strategy.py:470)
    mine.update(got, got_cost)
    assert mine.idxs_lb[np.asarray(got, dtype=np.int64)].all()
