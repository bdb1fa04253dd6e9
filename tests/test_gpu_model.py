"""End-to-end GPU tests of the public API and the model zoo."""
import os
import tempfile

import pytest
import torch

pytestmark = pytest.mark.gpu


class _ApiModel(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.e = torch.nn.Embedding(5000, 12)
        self.small = torch.nn.Embedding(10, 4)
        self.l = torch.nn.Linear(16, 1)

    def forward(self, x, y):
        return self.l(torch.cat([self.e(x), self.small(y)], -1)).squeeze(-1)


def _batch(vocab, B, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    ids = torch.stack([torch.randint(0, v, (B,), generator=g) for v in vocab], dim=1).to(dev)
    dense = torch.rand(B, 13, generator=g).to(dev)
    labels = (torch.rand(B, generator=g) < 0.3).float().to(dev)
    return ids, dense, labels


@pytest.mark.parametrize("name", ["lr", "wdl", "deepfm", "xdeepfm", "dcn"])
def test_models_train(cuda_context, name):
    from openembedding_b200.context import get_context
    from openembedding_b200.models.ctr import CTRModel
    from openembedding_b200.models.trainer import Trainer
    ctx = get_context()
    vocab = [1000, 50, 20000, 7, 3000] + [300] * 21
    torch.manual_seed(0)
    m = CTRModel(vocab, embedding_dim=9, model=name, batch=128, cache_threshold=64,
                 sparse_optimizer={"category": "adagrad", "learning_rate": 0.05})
    tr = Trainer(m, lr=0.05, use_graph=False)
    b = _batch(vocab, 128, ctx.device)
    losses = [float(tr.step(*b)) for _ in range(8)]
    ctx.backend.engine.check()
    assert losses[-1] < losses[0], losses


def test_graph_matches_eager(cuda_context):
    from openembedding_b200.context import get_context, reset_context
    from openembedding_b200.models.ctr import CTRModel
    from openembedding_b200.models.trainer import Trainer
    vocab = [1000, 50, 20000, 7, 3000] + [300] * 21
    res = []
    for graph in (False, True):
        reset_context()
        ctx = get_context()
        torch.manual_seed(0)
        m = CTRModel(vocab, embedding_dim=16, model="deepfm", batch=128, cache_threshold=0, compute_dtype=torch.float32)
        tr = Trainer(m, lr=0.01, use_graph=graph)
        ls = []
        if not graph:   # graph capture warms up with 3 real steps on the first batch; mirror that
            for _ in range(3):
                tr.step(*_batch(vocab, 128, ctx.device, seed=0))
        for s in range(6):
            ls.append(float(tr.step(*_batch(vocab, 128, ctx.device, seed=s))))
        ctx.backend.engine.check()
        res.append(ls)
    for a, b in zip(*res):
        assert abs(a - b) < 1e-3, res


class _CountingTrainer:
    """a trainer with next-batch prefetch that records which batch every step trains (the batch number is its ids)"""
    supports_prefetch = want_prefetch = True

    def __init__(self, device):
        self.device, self.trained = device, []

    def step(self, ids, dense, labels, next_ids=None, stable=False):
        self.trained.append(int(ids[0, 0]))
        return labels.sum()


def test_pipeline_trains_every_batch_once(cuda_context):
    """the one-batch-ahead input pipeline trains each submitted batch exactly once, also when last_loss() drains it
    between two runs of submits"""
    from openembedding_b200.models.trainer import _Pipeline
    tr = _CountingTrainer(torch.device("cuda", torch.cuda.current_device()))
    pipe = _Pipeline(tr, 4, 2, 1)

    def submit(k):
        pipe.submit(torch.full((4, 2), k, dtype=torch.int64).pin_memory(), torch.zeros(4, 1).pin_memory(),
                    torch.full((4,), float(k)).pin_memory())

    for k in range(5):
        submit(k)
    assert pipe.last_loss() == 4 * 4
    for k in range(5, 12):
        submit(k)
    assert pipe.last_loss() == 4 * 11
    assert tr.trained == list(range(12))


def test_api_embedding_checkpoint_roundtrip(cuda_context):
    import openembedding_b200.torch as embed
    from openembedding_b200.context import get_context
    M = _ApiModel
    m = embed.distributed_model(M())
    assert isinstance(m.e, embed.Embedding) and not m.e.sparse_as_dense and m.small.sparse_as_dense
    h = embed.Embedding(-1, 8, embeddings_initializer="uniform")
    ctx = get_context()
    opt = embed.distributed_optimizer(torch.optim.Adam(list(m.parameters()) + list(h.parameters()), lr=0.01))
    x = torch.randint(0, 5000, (300,), device=ctx.device)
    y = torch.randint(0, 10, (300,), device=ctx.device)
    t = torch.rand(300, device=ctx.device)
    l0 = None
    for i in range(10):
        loss = ((m(x, y) + h(x * 999983).sum(-1) - t) ** 2).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        l0 = l0 or float(loss)
    assert float(loss) < l0
    d = tempfile.mkdtemp()
    m.save_weights(d + "/ck")
    before_e, before_h = m.e(x).detach().clone(), h(x * 999983).detach().clone()
    for i in range(3):
        loss = ((m(x, y) + h(x * 999983).sum(-1) - t) ** 2).mean()
        opt.zero_grad(); loss.backward(); opt.step()
    assert float((m.e(x) - before_e).abs().max()) > 0
    m.load_weights(d + "/ck")
    assert torch.equal(m.e(x), before_e)
    assert torch.equal(h(x * 999983), before_h)
    # optimizer state survived: one more identical step from the restored state is deterministic
    plain = m.save_as_original_model(d + "/plain.pt")
    assert isinstance(plain.e, torch.nn.Embedding) and plain.e.weight.shape == (5000, 12)
    assert torch.allclose(plain.e.weight[x.cpu()], before_e.cpu())
    ctx.backend.engine.check()


def test_hash_table_grows_automatically():
    """a hashed Embedding whose shard starts tiny keeps training: the periodic maintenance tick doubles the
    shard before it fills up (reference: EasyHashMap rehash on insert)"""
    import openembedding_b200 as oe
    import openembedding_b200.torch as embed
    from openembedding_b200.context import get_context, reset_context
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    reset_context()
    old_dev, old_cfg = oe.flags.device, oe.flags.config
    oe.flags.device = "cuda"
    oe.flags.config = '{"server": {"hash_table_reserve": 256, "hash_table_grow_interval": 1}}'
    try:
        ctx = get_context()
        emb = embed.Embedding(-1, 8, embeddings_initializer={"category": "constant", "value": 0.0})
        opt = embed.distributed_optimizer(torch.optim.SGD(emb.parameters(), lr=1.0))
        seen = set()
        for step in range(12):
            ids = torch.arange(step * 100, step * 100 + 100, device=ctx.device) * 7919 + 13
            seen.update(ids.tolist())
            loss = emb(ids).sum()
            opt.zero_grad(); loss.backward(); opt.step()
        ctx.backend.engine.check()
        meta = emb.variable.variable
        assert ctx.backend.engine.table_size(meta.handle) == len(seen) == 1200
        assert ctx.backend.engine.table_info(meta.handle)["rows"] >= 2 * 1200     # grew from 256 slots
        probe = torch.tensor(sorted(seen)[:50], device=ctx.device)
        assert torch.allclose(emb(probe), torch.full((50, 8), -1.0, device=ctx.device))
    finally:
        oe.flags.device, oe.flags.config = old_dev, old_cfg
        reset_context()


class _WideModel(torch.nn.Module):
    """reference-style network script (examples/criteo_deepctr_network.py): nn.Embedding per sparse column,
    one [B, F] id matrix sliced by column inside forward, plus a keyword id tensor"""

    def __init__(self, vocab, dim):
        super().__init__()
        self.embs = torch.nn.ModuleList([torch.nn.Embedding(v, dim) for v in vocab])
        self.lin = torch.nn.ModuleList([torch.nn.Embedding(v, 1) for v in vocab])
        self.extra = torch.nn.Embedding(777, dim)
        self.mlp = torch.nn.Sequential(torch.nn.Linear(dim * (len(vocab) + 1), 32), torch.nn.ReLU(), torch.nn.Linear(32, 1))

    def forward(self, ids, extra=None):
        e = [m(ids[:, f]) for f, m in enumerate(self.embs)] + [self.extra(extra)]
        l = sum(m(ids[:, f]).squeeze(-1) for f, m in enumerate(self.lin))
        return self.mlp(torch.cat(e, dim=-1)).squeeze(-1) + l


def test_api_fused_group_matches_per_variable(cuda_context, monkeypatch):
    """distributed_model groups every server Embedding fed directly by a model input into ONE plan
    (one pull + one push+update launch per step); results are identical to the per-variable path"""
    import openembedding_b200.torch as embed
    from openembedding_b200.context import get_context, reset_context
    vocab = [5000, 300, 70000, 1200, 90]
    B = 192
    res = []
    for fused in ("0", "1"):
        monkeypatch.setenv("EXB_API_FUSED", fused)
        reset_context()
        ctx = get_context()
        torch.manual_seed(0)
        model = embed.distributed_model(_WideModel(vocab, 8), sparse_as_dense_size=100)
        opt = embed.distributed_optimizer(torch.optim.Adagrad(model.parameters(), lr=0.05, initial_accumulator_value=0.1))
        g = torch.Generator().manual_seed(3)
        losses = []
        for step in range(8):
            ids = torch.stack([torch.randint(0, v, (B,), generator=g) for v in vocab], 1).to(ctx.device)
            ex = torch.randint(0, 777, (B,), generator=g).to(ctx.device)
            y = (torch.rand(B, generator=g) < 0.3).float().to(ctx.device)
            loss = torch.nn.functional.binary_cross_entropy_with_logits(model(ids, extra=ex), y)
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(float(loss.detach()))
        ctx.backend.engine.check()
        model.eval()
        with torch.no_grad():
            probe = model(torch.stack([torch.arange(B) % v for v in vocab], 1).to(ctx.device),
                          extra=(torch.arange(B) % 777).to(ctx.device)).cpu()
        grp = getattr(model, "_embedding_group", None)
        res.append((losses, probe, grp))
    assert res[1][2] is not None and res[1][2].state == "on" and len(res[1][2].members) == 9, \
        (res[1][2].state, len(res[1][2].members))       # 4 + 4 server tables (vocab > 100) + extra
    assert res[0][0][-1] < res[0][0][0]
    for a, b in zip(res[0][0], res[1][0]):
        assert abs(a - b) < 1e-5, (res[0][0], res[1][0])
    assert torch.allclose(res[0][1], res[1][1], atol=1e-5)
