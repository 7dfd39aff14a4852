"""Edge cases of the reference semantics (SURVEY App. A), checked against the oracle on a small graph:
heads without rules, empty bodies only, relations without train edges, B = 1 / 33 / 64, arbitrary
(not the query's own) edges_to_remove, entities without out-edges, the empty-candidate quirks of
predictors.py:67-71 / 230-237."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def world():
    from rnnlogic_b200 import KnowledgeGraph
    from oracle import rnnlogic_oracle as O
    rng = np.random.default_rng(3)
    N, R = 90, 7                                   # relation 5 has NO train edge, relation 6 no rules
    tri = np.unique(np.stack([rng.integers(N - 10, size=700), rng.integers(5, size=700), rng.integers(N - 10, size=700)], 1), axis=0)
    tri = np.concatenate([tri, [[3, 6, 4], [5, 6, 7]]])
    rng.shuffle(tri)
    kg = KnowledgeGraph(entity_size=N, relation_size=R, train=tri, valid=tri[:20], test=tri[20:40])
    okg = O.OracleKG(N, R, tri, tri[:20], tri[20:40])
    rules = [[0, 1, 2], [0, 0], [0], [0, 5, 1], [0, 1, 5], [0, 0, 0, 0], [1], [1], [2, 3], [2, 3], [3, 5], [4, 2, 2, 2, 2, 2]]
    return kg, okg, rules, tri


def oracle_scores(okg, rules, w, bias, h, q, etr):
    from oracle import rnnlogic_oracle as O
    table = O.relation2rules(O.parse_rules(rules), okg.relation_size)
    return O.predictor_forward(okg, table[q], w, bias, torch.as_tensor(h), etr, q)


@pytest.mark.parametrize("ef", ["bias", "none"])
@pytest.mark.parametrize("B", [1, 33, 64])
def test_predictor_forward_matches_oracle(world, ef, B):
    from rnnlogic_b200.predictors import Predictor
    kg, okg, rules, tri = world
    g = torch.Generator().manual_seed(1)
    m = Predictor(kg, ef)
    m.set_rules(rules)
    with torch.no_grad():
        m.rule_weights.copy_(torch.randn(len(rules), generator=g))
        if ef == "bias":
            m.bias.copy_(torch.randn(kg.entity_size, generator=g))
    w = m.rule_weights.detach().clone()
    b = m.bias.detach().clone() if ef == "bias" else None
    m = m.cuda()
    rng = np.random.default_rng(B)
    for q in range(kg.relation_size):
        h = rng.integers(kg.entity_size, size=B)                  # includes entities 80..89 that have no edge at all
        n_q = int(okg.rel_ptr[q + 1] - okg.rel_ptr[q])
        for etr in (None, rng.integers(n_q, size=B) if n_q else None):   # ANY edge of relation q, not the query's own
            ht, rt = torch.from_numpy(h).to(DEV), torch.full((B,), q, device=DEV)
            with torch.no_grad():
                score, mask = m(ht, rt, None if etr is None else torch.from_numpy(etr).to(DEV))
            want, wmask = oracle_scores(okg, rules, w, b, h, q, etr)
            assert torch.equal(mask.cpu(), wmask), (q, ef)
            assert torch.equal(torch.isinf(score.cpu()), torch.isinf(want))
            fin = torch.isfinite(want)
            np.testing.assert_allclose(score.cpu()[fin].numpy(), want[fin].numpy(), rtol=1e-5, atol=1e-6)
            assert torch.equal(score.cpu()[~fin], want[~fin])      # same +/-inf pattern (predictors.py:71 quirk incl.)


def test_grounding_special_bodies(world):
    kg, okg, rules, tri = world
    h = torch.tensor([0, 5, 85, 3, 3])
    for q, body in ((0, []), (0, [5]), (0, [1, 5, 2]), (6, [6]), (6, [6, 6]), (2, [6, 0])):
        n_q = int(okg.rel_ptr[q + 1] - okg.rel_ptr[q])
        etr = torch.tensor([0, n_q - 1, 0, 0, n_q - 1]) if n_q else None
        got = kg.grounding(h.to(DEV), q, body, None if etr is None else etr.to(DEV)).cpu().numpy()
        want = okg.grounding(h.numpy(), q, body, None if etr is None else etr.numpy())
        assert np.array_equal(got, want), (q, body)


def test_compute_H_without_rules_and_plus_empty_case(world, tmp_path):
    from rnnlogic_b200.predictors import Predictor, PredictorPlus
    from oracle import rnnlogic_oracle as O
    kg, okg, rules, tri = world
    m = Predictor(kg, "bias")
    m.set_rules(rules)
    m = m.cuda()
    h = torch.tensor([3, 5], device=DEV)
    r = torch.full((2,), 6, device=DEV)
    assert m.compute_H(h, r, torch.tensor([4, 7], device=DEV), torch.tensor([0, 1], device=DEV)) == (None, None)
    for ef in ("bias", "none"):
        torch.manual_seed(0)
        pm = PredictorPlus(kg, type="emb", hidden_dim=16, entity_feature=ef, aggregator="sum")
        pm.set_rules(rules)
        pm = pm.cuda()
        score, mask = pm(h, r, None)                               # head 6 has no rule: predictors.py:230-237
        if ef == "bias":
            assert mask.all() and torch.equal(score, pm.bias.detach().unsqueeze(0).expand(2, -1))
        else:
            assert not mask.any() and torch.isinf(score).all() and (score > 0).all()
        # a normal head through the fused step still works with B = 1
        fact = [f for f in kg.train_facts if f[1] == 0][:1]
        loss, tsum = pm.fused_train_step([fact], 0.2)
        assert torch.isfinite(loss).all()


def test_wrong_inputs_raise(world):
    from rnnlogic_b200.predictors import Predictor, PredictorPlus
    from rnnlogic_b200 import _lib
    kg, okg, rules, tri = world
    m = Predictor(kg, "bias")
    with pytest.raises(ValueError):
        m.set_rules(3)
    m.set_rules(rules)
    m = m.cuda()
    with pytest.raises(AssertionError):                            # mixed relations in one batch (predictors.py:55)
        m(torch.tensor([1, 2], device=DEV), torch.tensor([0, 1], device=DEV), None)
    with pytest.raises(_lib.RlError):                              # CPU batch: no fallback
        m(torch.tensor([1, 2]), torch.tensor([0, 0]), None)
    with pytest.raises(NotImplementedError):
        PredictorPlus(kg, type="transformer")
    with pytest.raises(NotImplementedError):
        PredictorPlus(kg, aggregator="mean")


def test_device_lookup_of_the_removed_query_edge(world):
    """rl_prepare_slots(remove_query_edges): the query's own triple is masked iff it is a train edge -- same
    lanes as the host look-up of its per-relation index (data.py:214-216); triples that are not in train
    (and duplicates of a train triple) behave like the reference's index path."""
    from rnnlogic_b200.predictors import Predictor
    kg, okg, rules, tri = world
    m = Predictor(kg, "bias")
    m.set_rules(rules)
    m = m.cuda()
    sk = m._driver(torch.device(DEV))
    rng = np.random.default_rng(11)
    train_set = set(map(tuple, tri.tolist()))
    for q in range(5):
        own = tri[tri[:, 1] == q][:20]
        fake = np.stack([rng.integers(kg.entity_size, size=32 - len(own)), np.full(32 - len(own), q),
                         rng.integers(kg.entity_size, size=32 - len(own))], 1)
        batch = np.concatenate([own, fake]).astype(np.int64)              # 32 queries: train triples and random ones
        in_train = np.array([tuple(t) in train_set for t in batch.tolist()])
        assert in_train[:len(own)].all()
        idx = np.full(len(batch), -1, dtype=np.int64)                     # -1: no edge removed (not a train triple)
        idx[in_train] = kg.edge_index_of(batch[in_train])
        a = sk.gr.make_slots_host([batch], with_etr=True)                 # device look-up
        b = sk.gr.make_slots_host([batch], with_etr=True, etr_lists=[idx.tolist()])   # explicit reference indices
        assert torch.equal(a.lane.cpu(), b.lane.cpu()), q
    # end to end: the fused step equals the step driven by explicit indices
    batch = tri[tri[:, 1] == 0][:32].astype(np.int64)
    sl = sk.gr.make_slots_host([batch], with_etr=True)
    sk.gr.ground(sl)
    Za, _ = sk.predictor_scores(sl, m.rule_weights.detach(), m.bias.detach(), False)
    Za = Za.clone()
    sl2 = sk.gr.make_slots_host([batch], with_etr=True, etr_lists=[kg.edge_index_of(batch).tolist()])
    sk.gr.ground(sl2)
    Zb, _ = sk.predictor_scores(sl2, m.rule_weights.detach(), m.bias.detach(), False)
    assert torch.equal(Za, Zb)
