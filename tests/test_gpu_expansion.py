"""Frontier expansion cases the parity tests do not reach: a reused arena holding another call's rows, sparse and
all-rows nodes in one call on the typed graph, the removed query edge next to a parallel edge of another relation,
and a 32-bit row that only fits after the removed-edge fix-up."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _small_kg(N=60, R=3, E=1500, seed=0):
    from rnnlogic_b200 import KnowledgeGraph
    from oracle import rnnlogic_oracle as O
    rng = np.random.default_rng(seed)
    tri = np.unique(np.stack([rng.integers(N, size=E), rng.integers(R, size=E), rng.integers(N, size=E)], 1), axis=0)
    rng.shuffle(tri)
    kg = KnowledgeGraph(entity_size=N, relation_size=R, train=tri)
    okg = O.OracleKG(N, R, tri, np.zeros((0, 3), np.int64), np.zeros((0, 3), np.int64))
    return kg, okg, tri


def _queries(kg, tri, q, n, seed):
    rng = np.random.default_rng(seed)
    facts = tri[tri[:, 1] == q]
    facts = facts[rng.permutation(facts.shape[0])[:n]]
    return facts, kg.edge_index_of(facts)


def _ground(gr, q, facts, etr, workspace=False, check_overflow=True):
    sl = gr.make_slots([q], [facts.shape[0]], torch.from_numpy(facts[:, 0]).to(DEV), None, torch.from_numpy(etr).to(DEV))
    sl.use_workspace = workspace
    return gr.ground(sl, check_overflow=check_overflow)


@pytest.mark.parametrize("bits", [32, 64])
def test_reused_arena_is_never_read_stale(bits):
    """Call B on the same Grounder as call A (other heads, other queries) runs in a workspace arena that holds A's rows,
    then in one filled with garbage: its counts must equal a fresh Grounder's and the oracle's."""
    from rnnlogic_b200 import CompiledRules
    from rnnlogic_b200.engine import Grounder
    kg, okg, tri = _small_kg()
    rules = [(q, b) for q in range(3) for b in ([q], [1, q], [q, 2], [0, 1, q], [q, q, 0], [2, 2, 1, q])]
    cr = CompiledRules(kg, rules)
    gr = Grounder(kg, cr, DEV)
    fresh = Grounder(kg, cr, DEV)
    for g in (gr, fresh):
        g.force_bits = bits
    fa, ea = _queries(kg, tri, 0, 32, 1)
    _ground(gr, 0, fa, ea, workspace=True)
    fb, eb = _queries(kg, tri, 2, 32, 2)
    ids = cr.head_rules[2]
    want = np.stack([okg.grounding(fb[:, 0], 2, rules[i][1], eb) for i in ids])
    ref = fresh.rule_counts(_ground(fresh, 2, fb, eb), ids).cpu().numpy()
    assert np.array_equal(ref, want)
    for poison in (False, True):
        if poison:
            gr._ws_arena.fill_(0x5A5A5A5A)
        got = gr.rule_counts(_ground(gr, 2, fb, eb, workspace=True), ids).cpu().numpy()
        assert np.array_equal(got, want), poison


def test_removed_edge_on_parallel_edges_and_head_hops():
    """The query's own edge (h, q, t) is cut on every hop over q -- at depth 1 and 2, next to a parallel edge
    (h, r, t) of another relation that stays -- with sparse nodes only and with all-rows nodes only."""
    from rnnlogic_b200 import CompiledRules
    from rnnlogic_b200.engine import Grounder
    kg, okg, tri = _small_kg(N=40, R=3, E=1800, seed=3)
    q = 1
    pairs = set(map(tuple, tri[:, [0, 2]][tri[:, 1] != q]))
    facts = np.array([f for f in tri[tri[:, 1] == q] if (f[0], f[2]) in pairs][:32])
    assert facts.shape[0] >= 8
    etr = kg.edge_index_of(facts)
    bodies = [[q], [0, q], [q, q], [2, q], [q, 0], [q, q, q], [0, q, 2]]
    cr = CompiledRules(kg, [(q, b) for b in bodies])
    for num, den in ((1 << 20, 1), (0, 1)):               # never / always switch a node to all its rows
        gr = Grounder(kg, cr, DEV)
        gr.dense_num, gr.dense_den = num, den
        got = gr.rule_counts(_ground(gr, q, facts, etr), list(range(len(bodies)))).cpu().numpy()
        for i, b in enumerate(bodies):
            assert np.array_equal(got[i], okg.grounding(facts[:, 0], q, b, etr)), (num, b)


def test_fixup_brings_row_back_into_32bit():
    """A 32-bit row whose raw sum is 2^32 but whose count after the removed-edge fix-up is 3 * 2^30: the sum is kept in
    64 bits until the fix-up, so the 32-bit pass is exact and raises no overflow."""
    from rnnlogic_b200 import KnowledgeGraph, CompiledRules
    from rnnlogic_b200.engine import Grounder
    from oracle import rnnlogic_oracle as O
    w, k = 32, 6                                              # layered complete graph: 32^6 = 2^30 paths per entity
    h, q, r = 0, 0, 1
    layers = [list(range(1 + i * w, 1 + (i + 1) * w)) for i in range(k)]
    u = [1 + k * w + i for i in range(3)]
    t = 1 + k * w + 3
    N = t + 1
    tri = [(h, r, a) for a in layers[0]]
    for i in range(k - 1):
        tri += [(a, r, b) for a in layers[i] for b in layers[i + 1]]
    tri += [(a, r, b) for a in layers[-1] for b in u + [h]]
    tri += [(b, q, t) for b in u + [h]]
    tri = np.array(tri, dtype=np.int64)
    kg = KnowledgeGraph(entity_size=N, relation_size=2, train=tri)
    okg = O.OracleKG(N, 2, tri, np.zeros((0, 3), np.int64), np.zeros((0, 3), np.int64))
    body = [r] * (k + 1) + [q]
    facts = np.array([(h, q, t)], dtype=np.int64)
    etr = kg.edge_index_of(facts)
    want = okg.grounding(facts[:, 0], q, body, etr)
    assert want[0, t] == 3 << 30
    gr = Grounder(kg, CompiledRules(kg, [(q, body)]), DEV)
    gr.dense_num, gr.dense_den = 1 << 20, 1
    gr.force_bits = 32
    sl = _ground(gr, q, facts, etr, check_overflow=False)      # the 32-bit pass alone
    assert int(sl.overflow.item()) == 0
    assert np.array_equal(gr.rule_counts(sl, [0])[0].cpu().numpy(), want)


def test_typed_graph_mixes_sparse_and_all_rows_nodes():
    """Typed synthetic graph (FB15k-237 sizes): the dense switch gives some nodes of a call all their rows and keeps
    the others sparse.  Sparse == force_dense == oracle on sampled rules."""
    from rnnlogic_b200 import synth, KnowledgeGraph, CompiledRules
    from rnnlogic_b200.engine import Grounder
    from oracle import rnnlogic_oracle as O
    shape = synth.load_shape("fb15k237")
    N, R, train, valid, test, meta = synth.typed_kg(shape)
    rules = synth.typed_rules(shape, meta)
    kg = KnowledgeGraph(entity_size=N, relation_size=R, train=train, valid=valid, test=test)
    okg = O.OracleKG(N, R, train, valid[:0], test[:0])
    cr = CompiledRules(kg, rules)
    sparse, dense = Grounder(kg, cr, DEV), Grounder(kg, cr, DEV, force_dense=True)
    rec = cr.host["node_rec"].reshape(-1, 8)
    rng = np.random.default_rng(0)
    heads = [q for q in rng.permutation(R) if len(cr.head_rules[q]) >= 20][:3]
    n_all = n_sparse = 0
    for q in heads:
        facts, etr = _queries(kg, train, int(q), 32, int(q))
        s1, s2 = _ground(sparse, q, facts, etr), _ground(dense, q, facts, etr)
        # which nodes of the call took all their rows: parent with more than 1/4 of its rows non-zero
        n0, n1 = int(cr.head_node_ptr[q]), int(cr.head_node_ptr[q + 1])
        cnt = s1.state[s1.mask_words + 1:s1.mask_words + 1 + (n1 - n0)].cpu().numpy()
        for v in range(n0, n1):
            p = int(rec[v, 1])
            if cr.node_depth[v] >= 2 and cnt[p - n0] > 0:
                switched = cnt[p - n0] * sparse.dense_den > kg.rel_rows[rec[v, 2]] * sparse.dense_num
                n_all += int(switched)
                n_sparse += int(not switched)
        ids = cr.head_rules[q]
        longest = sorted(ids, key=lambda i: -len(rules[i][1]))[:4]
        pick = sorted(set(int(i) for i in rng.choice(ids, size=8, replace=False)) | set(longest))
        c1, c2 = sparse.rule_counts(s1, pick), dense.rule_counts(s2, pick)
        assert torch.equal(c1, c2)
        got = c1.cpu().numpy()
        for i, rid in enumerate(pick):
            assert np.array_equal(got[i], okg.grounding(facts[:, 0], q, rules[rid][1], etr)), (q, rid)
    assert n_all > 0 and n_sparse > 0, (n_all, n_sparse)
