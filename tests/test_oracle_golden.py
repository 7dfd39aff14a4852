"""Pin the CPU oracle (oracle/rnnlogic_oracle.py + grounding_oracle.c) against outputs of the
unmodified reference stored in tests/golden/ (made by tests/golden/make_golden.py).

Integer results (path counts, (L,H) rank bounds) must be bit-exact; fp32 results are compared
at rtol 1e-5 (north_star tolerance) with a small atol for values that cancel to ~0."""
import os

import numpy as np
import pytest
import torch

from tests import _golden as G
from oracle import rnnlogic_oracle as O

RTOL, ATOL = 1e-5, 2e-6


@pytest.fixture(scope="module", autouse=True)
def golden_thread_count():
    """The golden outputs were recorded with 8 intra-op threads.  torch splits a CPU reduction by its thread count, so a
    sum that cancels to ~0 (the gradient of the bias in front of the softmax) reproduces only at the same count."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def kg_of(fx):
    return O.OracleKG(int(fx["N"]), int(fx["R"]), fx["train"], fx["valid"], fx["test"])


@pytest.fixture(scope="module", params=G.DATASETS)
def ds(request):
    fx = G.load(request.param)
    kg = kg_of(fx)
    rules = O.parse_rules(G.rules_of(fx))
    return request.param, fx, kg, rules


def test_grounding_counts_bit_exact(ds):
    name, fx, kg, rules = ds
    n = int(fx["gr_n"])
    assert n > 20
    for c in range(n):
        tri, _, etr = G.train_batch_inputs(fx, int(fx["gr%d_batch" % c]))
        head, body = rules[int(fx["gr%d_rule" % c])]
        use = bool(fx["gr%d_etr" % c])
        got = kg.grounding(tri[:, 0], head, body, etr.numpy() if use else None)
        want = fx["gr%d_counts" % c]
        assert got.dtype == np.int64 and np.array_equal(got, want), (name, c)
        if c % 7 == 0:
            assert np.array_equal(kg.grounding_numpy(tri[:, 0], head, body, etr.numpy() if use else None), want)


def test_batch_builders(ds):
    name, fx, kg, rules = ds
    for j in range(int(fx["tb_n"])):
        tri, target, etr = G.train_batch_inputs(fx, j)
        h, r, t, tg, e = O.train_batch(kg, [tuple(x) for x in tri.tolist()])
        assert torch.equal(tg, target) and torch.equal(e, etr)
    for j in range(int(fx["vb_n"])):
        tri, flag = G.valid_batch_inputs(fx, j)
        h, r, t, fl = O.eval_batch(kg, [tuple(x) for x in tri.tolist()], "valid")
        assert torch.equal(fl, flag)


@pytest.mark.parametrize("ef", ["bias", "none"])
def test_predictor_forward_loss_grad(ds, ef):
    name, fx, kg, rules = ds
    table = O.relation2rules(rules, kg.relation_size)
    for j in range(5):
        if "pred_%s_tb%d_score" % (ef, j) not in fx:
            continue
        tri, target, etr = G.train_batch_inputs(fx, j)
        q = int(tri[0, 1])
        w = torch.from_numpy(fx["pred_%s_w" % ef].copy()).requires_grad_()
        b = torch.from_numpy(fx["pred_bias_b"].copy()).requires_grad_() if ef == "bias" else None
        score, mask = O.predictor_forward(kg, table[q], w, b, torch.from_numpy(tri[:, 0]), etr.numpy(), q)
        assert torch.equal(mask, torch.from_numpy(fx["pred_%s_tb%d_mask" % (ef, j)]))
        np.testing.assert_allclose(score.detach().numpy(), fx["pred_%s_tb%d_score" % (ef, j)], rtol=RTOL, atol=ATOL)
        if "pred_%s_tb%d_loss" % (ef, j) in fx:
            tgt = O.smoothed_target(target, torch.from_numpy(tri[:, 2]), 0.2)
            loss = O.ce_loss(score, mask, tgt)
            loss.backward()
            np.testing.assert_allclose(loss.item(), fx["pred_%s_tb%d_loss" % (ef, j)], rtol=RTOL)
            np.testing.assert_allclose(w.grad.numpy(), fx["pred_%s_tb%d_gw" % (ef, j)], rtol=1e-4, atol=1e-6)
            if ef == "bias":
                np.testing.assert_allclose(b.grad.numpy(), fx["pred_bias_tb%d_gb" % j], rtol=1e-4, atol=1e-7)
        if ef == "bias" and "pred_bias_tb%d_H" % j in fx:
            H, idx = O.predictor_compute_H(kg, table[q], w.detach(), tri[:, 0], tri[:, 2], etr.numpy(), q)
            assert np.array_equal(idx.numpy(), fx["pred_bias_tb%d_Hidx" % j])
            np.testing.assert_allclose(H.numpy(), fx["pred_bias_tb%d_H" % j], rtol=1e-4, atol=1e-6)
    for j in range(4):
        key = "pred_%s_vb%d_score" % (ef, j)
        if key not in fx:
            continue
        tri, flag = G.valid_batch_inputs(fx, j)
        q = int(tri[0, 1])
        w = torch.from_numpy(fx["pred_%s_w" % ef].copy())
        b = torch.from_numpy(fx["pred_bias_b"].copy()) if ef == "bias" else None
        score, mask = O.predictor_forward(kg, table[q], w, b, torch.from_numpy(tri[:, 0]), None, q)
        assert torch.equal(mask, torch.from_numpy(fx["pred_%s_vb%d_mask" % (ef, j)]))
        np.testing.assert_allclose(score.numpy(), fx[key], rtol=RTOL, atol=ATOL)


def test_predictor_plus_variants(ds):
    name, fx, kg, rules = ds
    table = O.relation2rules(rules, kg.relation_size)
    feats = O.rule_features(rules, kg.relation_size)
    for tag in G.plus_tags(fx):
        cfg = G.plus_cfg(fx, tag)
        for j in range(3):
            if "%s_tb%d_score" % (tag, j) not in fx:
                continue
            p = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in G.plus_state(fx, tag).items()}
            tri, target, etr = G.train_batch_inputs(fx, j)
            score, mask = O.plus_forward(kg, table[int(tri[0, 1])], feats, p, cfg,
                                         tri[:, 0], tri[:, 1], etr.numpy())
            assert torch.equal(mask, torch.from_numpy(fx["%s_tb%d_mask" % (tag, j)])), (name, tag, j)
            np.testing.assert_allclose(score.detach().numpy(), fx["%s_tb%d_score" % (tag, j)],
                                       rtol=1e-4, atol=1e-5, err_msg="%s %s %d" % (name, tag, j))
            if "%s_tb%d_loss" % (tag, j) in fx:
                tgt = O.smoothed_target(target, torch.from_numpy(tri[:, 2]), 0.2)
                loss = O.ce_loss(score, mask, tgt)
                loss.backward()
                np.testing.assert_allclose(loss.item(), fx["%s_tb%d_loss" % (tag, j)], rtol=RTOL)
                for pn, par in p.items():
                    key = "%s_tb%d_g_%s" % (tag, j, pn)
                    if key in fx:
                        assert par.grad is not None, pn
                        scale = max(1e-6, float(np.abs(fx[key]).max()))
                        np.testing.assert_allclose(par.grad.numpy(), fx[key], rtol=1e-3, atol=2e-4 * scale,
                                                   err_msg="%s %s %s" % (name, tag, pn))
        for j in range(2):
            key = "%s_vb%d_score" % (tag, j)
            if key not in fx:
                continue
            p = G.plus_state(fx, tag)
            tri, flag = G.valid_batch_inputs(fx, j)
            with torch.no_grad():
                score, mask = O.plus_forward(kg, table[int(tri[0, 1])], feats, p, cfg, tri[:, 0], tri[:, 1], None)
            assert torch.equal(mask, torch.from_numpy(fx["%s_vb%d_mask" % (tag, j)]))
            np.testing.assert_allclose(score.numpy(), fx[key], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("ef", ["bias", "none"])
def test_filtered_rank_and_metrics(ds, ef):
    """(L,H) rows captured from the reference's TrainerPredictor.evaluate + its logged metrics."""
    name, fx, kg, rules = ds
    table = O.relation2rules(rules, kg.relation_size)
    w = torch.from_numpy(fx["pred_%s_w" % ef].copy())
    b = torch.from_numpy(fx["pred_bias_b"].copy()) if ef == "bias" else None
    sizes = fx["eval_%s_batches" % ef]
    triples = fx["eval_%s_triples" % ef].astype(np.int64)
    want_rows = fx["eval_%s_rows" % ef]
    rows, off = [], 0
    for n in sizes:
        tri = triples[off:off + n]
        off += n
        h, r, t, flag = O.eval_batch(kg, [tuple(x) for x in tri.tolist()], "valid")
        q = int(tri[0, 1])
        score, mask = O.predictor_forward(kg, table[q], w, b, h, None, q)
        LH = O.filtered_rank(score, flag, mask, t)
        rows += [[int(a), int(bb), int(c), int(l), int(hh)] for (a, bb, c), (l, hh) in zip(tri.tolist(), LH.tolist())]
    got = np.array(rows, dtype=np.int64)
    # the reference walks the batches in DistributedSampler (shuffled) order: compare as multisets
    got = got[np.lexsort(got.T[::-1])]
    want_rows = want_rows[np.lexsort(want_rows.T[::-1])]
    assert np.array_equal(got[:, :3], want_rows[:, :3])
    # logits are fp32 sums in both code bases but near-ties may order differently by 1 ulp
    diff = (got[:, 3:] != want_rows[:, 3:]).any(axis=1).mean()
    assert diff <= 0.002, diff
    for expectation in (True, False):
        m = O.rank_metrics(want_rows, expectation)
        logged = fx["eval_%s_%d_logged" % (ef, expectation)]
        assert m["data"] == int(logged[0])
        np.testing.assert_allclose([m["hit1"], m["hit3"], m["hit10"], m["mr"], m["mrr"]], logged[1:], rtol=0, atol=6e-7)
        np.testing.assert_allclose(m["mrr"], fx["eval_%s_%d_mrr" % (ef, expectation)], rtol=1e-12)
        m2 = O.rank_metrics(got, expectation)
        np.testing.assert_allclose(m2["mrr"], m["mrr"], rtol=1e-5)


@pytest.mark.parametrize("name", G.DATASETS)
def test_oracle_rule_search_matches_the_reference_miner(name):
    """Row f4: the C restatement of rule_search / RuleMiner::search (oracle_mine_rules) reproduces, rule for rule and in
    the same order, what the reference's own miner binary code mines (tests/golden/mined_*.npz, made by
    tests/golden/make_mined_golden.py from oracle/_ref); UMLS / Kinship counts are the survey's 39,283 / 70,229."""
    fx = G.load(name)
    gold = dict(np.load(os.path.join(G.GOLDEN, "mined_%s.npz" % name)))
    want = [[int(v) for v in row if v >= 0] for row in gold["rules"]]
    got = O.mine_rules(fx["train"], int(fx["N"]), int(fx["R"]), int(gold["max_length"]))
    assert len(got) == len(want) == {"umls": 39283, "kinship": 70229}.get(name, len(want))
    assert got == want


def test_oracle_rule_search_edge_cases():
    """h == t gives the empty body; r <- r is dropped; the triple itself is removed wherever it occurs; a path stops
    at its first visit of t."""
    #        0 -r0-> 1 -r1-> 2,  0 -r2-> 2,  2 -r0-> 2 (self loop),  2 -r1-> 0
    train = np.array([[0, 0, 1], [1, 1, 2], [0, 2, 2], [2, 0, 2], [2, 1, 0]])
    rules = O.mine_rules(train, 3, 3, 3)
    assert [0] in rules                                   # (2, r0, 2): h == t
    assert [2, 0, 1] in rules                             # (0, r2, 2) via 0 -r0-> 1 -r1-> 2
    assert [2, 2] not in rules and [0, 0] not in rules    # trivial rules never appear
    assert [1, 1] not in rules
    # (0, r0, 1): 0 -r2-> 2 -r1-> 0 -r0-> 1 would use the removed triple; nothing else reaches 1
    assert not any(r[0] == 0 and len(r) > 1 for r in rules)
    # a path does not run THROUGH its goal: (1, r1, 2) has 2 -r0-> 2 behind the goal, never used
    assert all(r != [1, 1, 0] for r in rules)
