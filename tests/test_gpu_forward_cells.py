"""forward(all_h, all_r, edges_to_remove) of Predictor / PredictorPlus on the candidate cells: calls that are alive
together, cell arrays that have to grow, and the PredictorPlus shapes the cell kernels do not take (hidden_dim != 16)
against the oracle."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def world():
    from rnnlogic_b200 import KnowledgeGraph
    from oracle import rnnlogic_oracle as O
    rng = np.random.default_rng(17)
    N, R = 120, 6
    tri = np.unique(np.stack([rng.integers(N, size=1500), rng.integers(R, size=1500), rng.integers(N, size=1500)], 1), axis=0)
    rng.shuffle(tri)
    kg = KnowledgeGraph(entity_size=N, relation_size=R, train=tri, valid=tri[:20], test=tri[20:40])
    okg = O.OracleKG(N, R, tri, tri[:20], tri[20:40])
    rules = []
    for q in range(R):
        rules += [[q], [q, q], [q, q]]                                # empty body, duplicate rules
        rules += [[q] + [int(x) for x in rng.integers(R, size=int(rng.integers(1, 4)))] for _ in range(6)]
    return kg, okg, rules, tri


def batch_of(kg, tri, q, B):
    b = tri[tri[:, 1] == q][:B].astype(np.int64)
    t = torch.from_numpy(b).to(DEV)
    return b, t[:, 0], t[:, 1], torch.from_numpy(np.asarray(kg.edge_index_of(b), dtype=np.int64)).to(DEV)


def ce(score, mask, all_t, seed):
    """log(softmax + 1e-8) cross-entropy against a smoothed target (trainer.py:84,88-89)."""
    g = torch.Generator().manual_seed(seed)
    multi = (torch.rand(score.shape, generator=g) < 0.05).float().to(score.device)
    tgt = 0.2 * multi + 0.8 * torch.nn.functional.one_hot(all_t, score.shape[1]).to(score.dtype)
    lp = (torch.softmax(score, dim=1) + 1e-8).log()
    return -(lp[mask] * tgt[mask]).sum() / torch.clamp(tgt[mask].sum(), min=1)


def make(world, kind, ef, seed=0):
    from rnnlogic_b200.predictors import Predictor, PredictorPlus
    kg, okg, rules, tri = world
    torch.manual_seed(seed)
    if kind == "pred":
        m = Predictor(kg, ef)
    else:
        typ, agg = kind.split("+")
        m = PredictorPlus(kg, type=typ, num_layers=2, hidden_dim=16, entity_feature=ef, aggregator=agg)
    m.set_rules(rules)
    with torch.no_grad():
        if kind == "pred":
            m.rule_weights.copy_(torch.randn(len(rules)) * 0.3)
        if ef == "bias":
            m.bias.copy_(torch.randn(kg.entity_size) * 0.3)
    return m.cuda()


def grads(m):
    return {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}


def assert_same_grads(a, b):
    assert a.keys() == b.keys()
    for n in a:
        scale = max(1e-6, float(b[n].abs().max()))
        np.testing.assert_allclose(a[n].cpu().numpy(), b[n].cpu().numpy(), rtol=1e-5, atol=max(1e-6 * scale, 1e-7),
                                   err_msg=n)                        # a gradient that cancels to ~0 (mask mode: the MLP's last bias)


@pytest.mark.parametrize("kind,ef", [("pred", "bias"), ("pred", "none"), ("emb+sum", "bias"), ("lstm+pna", "none")])
def test_two_live_forward_calls(world, kind, ef):
    """Two forward() calls before one backward() of their summed losses == the same calls one after another (their
    gradients summed here: the LSTM encoder hands bias_ih and bias_hh one gradient tensor, so .grad must not
    accumulate over two backward() calls)."""
    kg, okg, rules, tri = world
    m = make(world, kind, ef)
    _, h1, r1, e1 = batch_of(kg, tri, 0, 40)                         # two slots
    _, h2, r2, e2 = batch_of(kg, tri, 3, 20)
    s1, k1 = m(h1, r1, e1)
    s2, k2 = m(h2, r2, e2)
    (ce(s1, k1, torch.from_numpy(tri[tri[:, 1] == 0][:40, 2]).to(DEV), 1)
     + ce(s2, k2, torch.from_numpy(tri[tri[:, 1] == 3][:20, 2]).to(DEV), 2)).backward()
    together = grads(m)
    outs, apart = [], {}
    for (h, r, e), q, B, seed in (((h1, r1, e1), 0, 40, 1), ((h2, r2, e2), 3, 20, 2)):
        m.zero_grad()
        s, k = m(h, r, e)
        ce(s, k, torch.from_numpy(tri[tri[:, 1] == q][:B, 2]).to(DEV), seed).backward()
        outs.append((s.detach(), k))
        for n, g in grads(m).items():
            apart[n] = apart[n] + g if n in apart else g
    for (s, k), (sa, ka) in zip(outs, ((s1.detach(), k1), (s2.detach(), k2))):
        assert torch.equal(k, ka)
        np.testing.assert_allclose(sa.cpu().numpy(), s.cpu().numpy(), rtol=1e-6, atol=1e-6)
    assert_same_grads(together, apart)


@pytest.mark.parametrize("kind,ef", [("pred", "bias"), ("emb+pna", "bias"), ("emb+sum", "none")])
def test_forward_with_growing_cell_arrays(world, kind, ef):
    """A call whose cells do not fit the first guess of the arrays is expanded again and built with the exact count."""
    kg, okg, rules, tri = world
    b, h, r, e = batch_of(kg, tri, 1, 40)
    t = torch.from_numpy(b[:, 2]).to(DEV)
    out = []
    for hint in (None, 1):
        m = make(world, kind, ef)
        gr = m._driver(torch.device(DEV)).gr
        caps = []
        build = gr.build_cells

        def counting_build(sl, floats, cap=None):
            caps.append(cap)
            return build(sl, floats, cap=cap)

        gr.build_cells = counting_build
        if hint is not None:
            gr.cells_per_slot_hint = hint
        s, k = m(h, r, e)
        ce(s, k, t, 3).backward()
        assert len(caps) == (1 if hint is None else 2)
        out.append((s.detach(), k, grads(m)))
    (s0, k0, g0), (s1, k1, g1) = out
    assert torch.equal(k0, k1)
    np.testing.assert_allclose(s1.cpu().numpy(), s0.cpu().numpy(), rtol=1e-6, atol=1e-6)
    assert_same_grads(g1, g0)


@pytest.mark.parametrize("H", [8, 32])
@pytest.mark.parametrize("agg", ["sum", "pna"])
@pytest.mark.parametrize("ef", ["bias", "none"])
def test_plus_generic_shapes_match_oracle(world, H, agg, ef):
    """PredictorPlus.forward at the widths the cell kernels do not take: scores, mask, loss and every parameter
    gradient against oracle.plus_forward (tolerances of test_gpu_plus)."""
    from rnnlogic_b200 import cellpath
    from rnnlogic_b200.predictors import PredictorPlus
    from oracle import rnnlogic_oracle as O
    kg, okg, rules, tri = world
    torch.manual_seed(H)
    m = PredictorPlus(kg, type="emb", hidden_dim=H, entity_feature=ef, aggregator=agg)
    m.set_rules(rules)
    if ef == "bias":
        with torch.no_grad():
            m.bias.copy_(torch.randn(kg.entity_size) * 0.3)
    p = {n: v.detach().clone().requires_grad_() for n, v in m.named_parameters()}
    m = m.cuda()
    assert not cellpath.plus_cells_supported(m)
    table = O.relation2rules(O.parse_rules(rules), kg.relation_size)
    cfg = dict(type="emb", num_layers=3, hidden_dim=H, entity_feature=ef, aggregator=agg)
    for q, B in ((0, 40), (2, 7)):
        b, h, r, e = batch_of(kg, tri, q, B)
        t = torch.from_numpy(b[:, 2])
        m.zero_grad()
        for v in p.values():
            v.grad = None
        score, mask = m(h, r, e)
        want, wmask = O.plus_forward(okg, table[q], None, p, cfg, b[:, 0], b[:, 1], e.cpu().numpy())
        assert torch.equal(mask.cpu(), wmask.bool()), (q, H, agg, ef)
        assert torch.equal(torch.isinf(score.detach().cpu()), torch.isinf(want.detach()))
        fin = torch.isfinite(want.detach())
        np.testing.assert_allclose(score.detach().cpu()[fin].numpy(), want.detach()[fin].numpy(), rtol=1e-4, atol=1e-5)
        loss = ce(score, mask, t.to(DEV), q)
        wloss = ce(want, wmask.bool(), t, q)
        loss.backward()
        wloss.backward()
        np.testing.assert_allclose(loss.item(), wloss.item(), rtol=1e-5)
        seen = 0
        for n, par in m.named_parameters():
            if p[n].grad is None:
                assert par.grad is None or not par.grad.any(), n
                continue
            want_g = p[n].grad.numpy()
            got = par.grad.cpu().numpy()
            scale = max(1e-6, float(np.abs(want_g).max()))
            err = np.abs(got - want_g)
            ok = err <= np.maximum(1e-4 * scale, 2e-7) + 1e-3 * np.abs(want_g)
            msg = "%s H%d %s %s q%d: %d/%d outside, max err %.3e (scale %.3e)" % (n, H, agg, ef, q, (~ok).sum(), ok.size, err.max(), scale)
            assert ok.all(), msg
            assert err.max() <= max(5e-2 * scale, 2e-7), msg
            seen += 1
        assert seen >= 4
