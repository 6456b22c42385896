"""Shared test scaffolding: a lookup "network"/dataset that lets tests choose the logits and
embeddings of every pool index, and OracleEngine -- an implementation of the Engine protocol on
CPU tensors built from oracle/al_oracle.py.  OracleEngine exists ONLY so the CPU test tier can
exercise the samplers' host logic (index bookkeeping, RNG order, partition batching, sharding);
it is never importable from the product package."""
import os
import tempfile

import numpy as np
import torch
import torch.nn as nn

from oracle import al_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden.npz")


def c1000_logits():
    """The 700 x 1000 logits of the f32_c1000 margin case (2.8 MB, too large to store).  make_golden.py drew them
    from torch's CPU generator seeded with 0, after the f32_c10 logits and the one int64 seed that case's DataLoader
    drew; this replays the same draws."""
    g = torch.Generator().manual_seed(0)
    torch.randn(700, 10, generator=g)
    torch.empty((), dtype=torch.int64).random_(generator=g)
    return torch.randn(700, 1000, generator=g) * 3.0


def load_gold(path=GOLD):
    """reference_golden.npz as a dict, with margin_f32_c1000_logits regenerated and checked against the strided
    sample make_golden.py stored of it."""
    gold = dict(np.load(path))
    logits = c1000_logits().numpy()
    assert np.array_equal(logits[::7, ::13], gold.pop("margin_f32_c1000_logits_sample")), \
        "torch's CPU generator no longer reproduces the f32_c1000 logits"
    gold["margin_f32_c1000_logits"] = logits
    return gold


class IndexDataset(torch.utils.data.Dataset):
    def __init__(self, n, num_classes):
        self.n, self.num_classes = n, num_classes
        self.targets = [0] * n

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        return torch.tensor(float(i)), 0, i


class LabeledIndexDataset(torch.utils.data.Dataset):
    """Pool stand-in whose labels matter (BalancingSampler reads y from the loader)."""

    def __init__(self, ys, num_classes):
        self.ys, self.num_classes = [int(v) for v in ys], num_classes
        self.targets = self.ys

    def __len__(self):
        return len(self.ys)

    def __getitem__(self, i):
        return torch.tensor(float(i)), self.ys[i], i


class LookupNet(nn.Module):
    """net(x) -> logits[x];  net(x, return_features=...) -> (logits[x], emb[x])."""

    def __init__(self, logits, emb):
        super().__init__()
        self.register_buffer("logits", logits.clone())
        self.register_buffer("emb", emb.clone())
        self.dummy = nn.Parameter(torch.zeros(1))

    def forward(self, x, return_features=False, specify_input_layer=None):
        i = x.long()
        if return_features:
            return self.logits[i], self.emb[i]
        return self.logits[i]


class HeadNet(nn.Module):
    """Embedding table + the linear head of the reference's models (resnet_simclr.py:21,29-41):
    logits = linear(emb[x]); `specify_input_layer="finalembed"` applies the head alone."""

    def __init__(self, emb, weight, bias):
        super().__init__()
        self.register_buffer("emb", emb.clone())
        self.linear = nn.Linear(weight.shape[1], weight.shape[0])
        with torch.no_grad():
            self.linear.weight.copy_(weight)
            self.linear.bias.copy_(bias)

    def forward(self, x, return_features=False, specify_input_layer=None):
        if specify_input_layer:
            assert specify_input_layer == "finalembed"
            return self.linear(x)
        h = self.emb[x.long()]
        out = self.linear(h)
        return (out, h) if return_features else out


class FakeExperiment:
    url = "."

    def get_key(self):
        return "test"

    def __getattr__(self, name):
        return lambda *a, **k: None


def make_strategy(name, logits, emb, eval_idxs, labeled, batch_size, engine=None, net=None, dataset=None, **kw):
    from active_learning_b200.query_strategies.get_strategy import get_strategy
    if net is None:
        n, c = logits.shape
        net = LookupNet(logits, emb)
    else:                                   # a HeadNet: logits come out of its own linear head
        n, c = net.emb.shape[0], net.linear.out_features
    ds = IndexDataset(n, c) if dataset is None else dataset
    args = dict(early_stop_patience=0, n_epoch=1, world_size=1, model="SSLResNet18",
                freeze_feature=True, ckpt_path=tempfile.mkdtemp(prefix="alq_test_"), exp_name="t",
                subset_labeled=None, subset_unlabeled=None, partitions=1)
    args.update(kw)
    train_args = {"loader_te_args": {"batch_size": batch_size, "num_workers": 0}}
    s = get_strategy(name)(ds, ds, net, train_args, np.array(eval_idxs, dtype=np.int64),
                           FakeExperiment(), None, **args)
    s.init_network_weights()
    if engine is not None:
        s.set_engine(engine)
    if len(labeled):
        s.update(np.array(labeled), len(labeled))
    return s


class OracleEngine:
    """Engine protocol on CPU tensors, arithmetic by the oracle."""
    device = torch.device("cpu")
    launches = 0

    def score_softmax(self, logits, mode, out=None):
        return O.softmax_scores(logits, mode, batch_size=128)

    def select_smallest(self, scores, b):
        return torch.from_numpy(O.select_smallest(scores, int(b)).astype(np.int32))

    def topb_pack(self, scores, pos, row_lo, b_pad, out=None):
        s = (scores.numpy().astype(np.float32) + np.float32(0.0)).view(np.uint32).astype(np.uint64)
        neg = (s >> np.uint64(31)).astype(bool)
        s = np.where(neg, ~s & np.uint64(0xFFFFFFFF), s | np.uint64(0x80000000))
        p = pos.numpy().astype(np.int64)
        words = np.full(int(b_pad), np.uint64(0xFFFFFFFFFFFFFFFF), dtype=np.uint64)
        words[:len(p)] = (s[p] << np.uint64(32)) | (p + int(row_lo)).astype(np.uint64)
        t = torch.from_numpy(words.view(np.int64).copy())
        if out is not None:
            out.copy_(t)
            return out
        return t

    def topb_merge(self, keys, b, list_len=0):
        w = np.sort(keys.numpy().view(np.uint64))[:int(b)]
        return torch.from_numpy((w & np.uint64(0xFFFFFFFF)).astype(np.int64).astype(np.int32))

    def badge_factors(self, logits, batch_size, row0=0, n_total=0):
        if n_total and (row0 or n_total != logits.shape[0]):
            # a shard [row0, row0 + n) of a loader pass over n_total rows: 1/bs of the GLOBAL batch each row falls in
            # (same closed form as O.badge_factors, badge_sampler.py:33-37)
            n, bsz = logits.shape[0], int(batch_size)
            g = np.arange(row0, row0 + n)
            tail = n_total % bsz
            bs_glob = np.where((tail > 0) & (g >= n_total - tail), tail, bsz).astype(np.float32)
            lg = logits.detach().to(torch.float32).cpu()
            onehot = torch.nn.functional.one_hot(lg.max(dim=1).indices, lg.shape[1]).to(torch.float32)
            a = (torch.softmax(lg, dim=1) - onehot) / torch.from_numpy(bs_glob)[:, None]
        else:
            a = O.badge_factors(logits, int(batch_size))
        cpad = (a.shape[1] + 3) & ~3
        ap = torch.zeros((a.shape[0], cpad))
        ap[:, :a.shape[1]] = a
        return ap, ap.square().sum(dim=1)

    def badge_pooled_embedding(self, logits, emb, batch_size):
        return O.gradient_embeddings(logits, emb, int(batch_size), use_adaptive_pool=True)

    def row_norm2(self, x):
        return x.square().sum(dim=1)

    def min_dist(self, x, xn, y, yn, xa=None, xan=None, ya=None, yan=None, reduce_max=False,
                 out=None, accumulate=False):
        dot = x @ y.T
        nx, ny = xn, yn
        if xa is not None:
            dot = dot * (xa @ ya.T)
            nx, ny = xn * xan, yn * yan
        d = (nx[:, None] + ny[None, :]) - 2 * dot
        r = d.max(dim=1).values if reduce_max else d.min(dim=1).values
        if out is not None:
            out.copy_(torch.maximum(out, r) if (accumulate and reduce_max) else
                      torch.minimum(out, r) if accumulate else r)
            return out
        return r

    def argmin(self, v):
        return int(v.min(dim=0).indices.item())

    def ratio_argmin(self, num, den, avail):
        r = (torch.ones_like(den) if num is None else num) / den
        r = torch.where(avail.bool(), r, torch.tensor(float("inf")))
        return int(r.min(dim=0).indices)

    def class_gap_inv(self, weight):
        w = weight.detach().float()
        den = ((w[:, None, :] - w[None, :, :]) ** 2).sum(dim=2)
        g = 1.0 / den.sqrt()
        g.fill_diagonal_(float("inf"))
        return g, torch.cat([g.min(dim=1).values, torch.ones(1)])

    def mase_margins(self, logits, gap, want_per_class=False):
        ginv = gap[0]
        pred = logits.max(dim=1).indices
        r = (logits.gather(1, pred[:, None]) - logits).abs() * ginv[pred][:, :logits.shape[1]]
        r = torch.where(torch.isnan(r), torch.tensor(float("inf")), r)
        r[torch.arange(len(r)), pred] = float("inf")
        return r.min(dim=1).values, pred.to(torch.int32), (r if want_per_class else None)

    def base_select(self, min_margin, radius, pred, budget):
        return torch.from_numpy(O.base_select(min_margin, radius, pred.long(), int(budget), radius.shape[1]).astype(np.int32))

    def greedy_select(self, x, xn, mind, part_off, budget, a=None, an=None, uniforms=None, vpos=None,
                      full_n=None, first_pick=None, variant=0, time_steps=False, shard_off=None, shard_pos=None):
        if shard_off is not None:
            # multi-rank protocol: arrays are global and replicated, every rank owns mind[shard]; the oracle engine
            # simply gathers the shards of `mind` and runs the whole loop on every rank
            import torch.distributed as dist
            world, rank = dist.get_world_size(), dist.get_rank()
            parts = [None] * world
            dist.all_gather_object(parts, mind[int(shard_off[rank]):int(shard_off[rank + 1])].clone())
            mind = torch.cat(parts)
            if shard_pos is not None:      # leaf-aligned shards: every rank's rows lie inside its position range
                vp = vpos.numpy()
                for r in range(world):
                    seg = vp[int(shard_off[r]):int(shard_off[r + 1])]
                    assert len(seg) == 0 or (seg.min() >= shard_pos[r] and seg.max() < shard_pos[r + 1])
        picks, u_at = [], 0
        nn_ = xn if a is None else xn * an
        for p in range(len(budget)):
            lo, hi, b = int(part_off[p]), int(part_off[p + 1]), int(budget[p])
            m = mind[lo:hi].clone()
            taken = np.zeros(hi - lo, dtype=bool)
            for t in range(b):
                if t == 0 and first_pick is not None and first_pick[p] >= 0:
                    q = int(first_pick[p]) - lo
                elif uniforms is None:
                    mm = m.clone()
                    mm[torch.from_numpy(taken)] = float("-inf")
                    q = int(mm.max(dim=0).indices.item())
                else:
                    full = np.zeros(int(full_n[p]), dtype=np.float32)
                    lab = np.ones(int(full_n[p]), dtype=bool)
                    vp = vpos[lo:hi].numpy()
                    full[vp] = m.numpy()
                    lab[vp] = taken
                    with np.errstate(invalid="ignore"):
                        k = O.d2_sampling_step(full, lab, float(uniforms[u_at + t]))
                    q = int(np.flatnonzero(vp == k)[0])
                picks.append(lo + q)
                taken[q] = True
                dot = x[lo:hi] @ x[lo + q]
                if a is not None:
                    dot = dot * (a[lo:hi] @ a[lo + q])
                m = torch.minimum(m, (nn_[lo:hi] + nn_[lo + q]) - 2 * dot)
            u_at += b
        mind.copy_(mind)
        out = np.asarray(picks, dtype=np.int32)
        return (out, 0.0) if time_steps else out
