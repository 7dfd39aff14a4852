"""CPU tests (no GPU): the C-ABI library loads and exports every symbol the header declares, the
host-side graph / rule compilers build what the kernels expect, and the multi-process pieces
(batch sharding, flat gradient all-reduce, rank-row gather) work at world size 2 over gloo."""
import os
import re

import numpy as np
import pytest
import torch

from tests import _golden as G


def test_cabi_library_exports_every_declared_symbol():
    from rnnlogic_b200 import _lib
    import ctypes
    header = open(os.path.join(G.ROOT, "include", "rnnlogic_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(rl_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    assert os.path.exists(_lib.LIB_PATH), "build with __graft_entry__.build()"
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(L, name), "missing export " + name
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())
    assert _lib.lib().rl_abi_version() == 5
    if not torch.cuda.is_available():           # no compute without a GPU -- and no silent fallback
        assert _lib.lib().rl_device_count() < 0
        assert b"no CPU fallback" in _lib.lib().rl_last_error()


def brute_rows(train, R):
    rows = {}
    for h, r, t in train.tolist():
        rows.setdefault((r, t), []).append(h)
    return rows


@pytest.mark.parametrize("name", G.DATASETS)
def test_graph_dcsr_matches_brute_force(name):
    from rnnlogic_b200 import KnowledgeGraph
    fx = G.load(name)
    N, R = int(fx["N"]), int(fx["R"])
    kg = KnowledgeGraph(entity_size=N, relation_size=R, train=fx["train"], valid=fx["valid"], test=fx["test"])
    H = kg.host
    rows = brute_rows(fx["train"].astype(np.int64), R)
    W = kg.rank_words
    rank = H["rank_tab"].reshape(R * W, 2)
    srank = H["srank_tab"].reshape(R * W, 2)
    assert H["row_dst"].shape[0] == len(rows)
    for r in range(R):
        for k in range(H["dst_ptr"][r], H["dst_ptr"][r + 1]):
            t = int(H["row_dst"][k])
            srcs = H["edge_src"][H["row_start"][k]:H["row_start"][k + 1]].tolist()
            assert sorted(srcs) == sorted(rows[(r, t)])
            bits, pre = rank[r * W + (t >> 5)]
            assert (int(bits) >> (t & 31)) & 1
            assert int(pre) + bin(int(bits) & ((1 << (t & 31)) - 1)).count("1") == k - H["dst_ptr"][r]
    # forward DCSR: every out-edge points at the local row of its tail
    for r in range(R):
        for k in range(H["fsrc_ptr"][r], H["fsrc_ptr"][r + 1]):
            for e in range(H["frow_start"][k], H["frow_start"][k + 1]):
                t = int(H["row_dst"][H["dst_ptr"][r] + H["fedge_dstrow"][e]])
                assert (r, t) in rows
    assert H["frow_start"][-1] == fx["train"].shape[0] and int(np.bitwise_count(srank[:, 0]).sum()) == H["fsrc_ptr"][-1]
    # reference edge order + edges_to_remove lookup (data.py:66-69, 214-216)
    ht = kg.relation2ht2index
    idx = kg.edge_index_of(fx["train"])
    for (h, r, t), k in list(zip(fx["train"].tolist(), idx.tolist()))[::37]:
        assert ht[r][kg.encode_ht(h, t)] == k
        assert H["ord_h"][H["ord_ptr"][r] + k] == h and H["ord_t"][H["ord_ptr"][r] + k] == t
    with pytest.raises(KeyError):
        kg.edge_index_of(np.array([[0, 0, 0]]) if (0, 0, 0) not in set(map(tuple, fx["train"].tolist())) else np.array([[N - 1, 0, N - 1]]))
    # answer lists == the reference dicts, de-duplicated
    for which in ("hr2o", "hr2oo", "hr2ooo"):
        keys, ptr, ent = kg.answers_csr(which)
        d = getattr(kg, which)
        assert sorted(d.keys()) == keys.tolist()
        for i in range(0, len(keys), 23):
            assert sorted(set(d[int(keys[i])])) == ent[ptr[i]:ptr[i + 1]].tolist()


def test_rule_compiler_tries():
    from rnnlogic_b200 import KnowledgeGraph, CompiledRules, parse_rules
    fx = G.load("umls")
    kg = KnowledgeGraph(entity_size=int(fx["N"]), relation_size=int(fx["R"]), train=fx["train"])
    full = parse_rules(G.rules_of(fx, "mined_rules"))
    cr = CompiledRules(kg, full)
    assert len(full) == 39283 and cr.num_nodes == 42956          # SURVEY.md section 7 step 2 (UMLS mined rules)
    rules = parse_rules(G.rules_of(fx))
    cr = CompiledRules(kg, rules)
    H = cr.host
    prefixes = set()
    for h, b in rules:
        for k in range(1, len(b) + 1):
            prefixes.add((h,) + tuple(b[:k]))
    assert cr.num_nodes == len(prefixes)
    # every rule end is the node spelled by walking parents back to the root
    for rid in range(0, len(rules), 11):
        node = int(cr.rule_node[rid])
        body = []
        while node >= 0:
            body.append(int(H["node_rel"][node]))
            node = int(H["node_parent"][node])
        assert body[::-1] == list(rules[rid][1])
    # chunks tile every node exactly once; depth ranges are contiguous
    rows = kg.rel_rows[H["node_rel"]]
    covered = np.zeros(cr.num_nodes, dtype=np.int64)
    np.add.at(covered, H["chunk_node"], np.minimum(32, rows[H["chunk_node"]] - H["chunk_row0"]))
    assert np.array_equal(covered, rows)
    assert cr.level_chunks.sum() == cr.num_chunks and cr.level_nodes.sum() == cr.num_nodes
    assert sum(len(b) == 0 for _, b in rules) == H["zr_ptr"][-1]
    with pytest.raises(ValueError):
        CompiledRules(kg, [(0, [kg.relation_size])])
    with pytest.raises(ValueError):
        parse_rules(3.5)


def test_datasets_follow_reference_random_order():
    """Same python-random call order as src/data.py:186-196, 232-238 => same batches as the golden run."""
    import random
    from rnnlogic_b200.data import KnowledgeGraph, TrainDataset, ValidDataset, TestDataset
    fx = G.load("umls")
    kg = KnowledgeGraph(entity_size=int(fx["N"]), relation_size=int(fx["R"]), train=fx["train"], valid=fx["valid"], test=fx["test"])
    random.seed(1)
    np.random.seed(1)
    torch.manual_seed(1)
    tr, va, te = TrainDataset(kg, 32), ValidDataset(kg, 32), TestDataset(kg, 32)
    got = set(tuple(map(tuple, b)) for b in tr.batches)
    for j in range(int(fx["tb_n"])):
        assert tuple(map(tuple, fx["tb%d_triples" % j].tolist())) in got
    tri, target, etr = G.train_batch_inputs(fx, 0)
    i = [k for k, b in enumerate(tr.batches) if tuple(map(tuple, b)) == tuple(map(tuple, tri.tolist()))][0]
    item = tr[i]
    assert torch.equal(item[3], target) and torch.equal(item[4], etr)
    tri, flag = G.valid_batch_inputs(fx, 0)
    i = [k for k, b in enumerate(va.batches) if tuple(map(tuple, b)) == tuple(map(tuple, tri.tolist()))][0]
    assert torch.equal(va[i][3], flag)


def test_shard_indices_is_distributed_sampler():
    from rnnlogic_b200.trainer import shard_indices, dedup_weights
    a, b = shard_indices(11, 2, 0), shard_indices(11, 2, 1)
    assert len(a) == len(b) == 6 and set(a) | set(b) == set(range(11))      # padded by wrap-around
    assert shard_indices(11, 1, 0) == shard_indices(11, 1, 0) and sorted(shard_indices(11, 1, 0)) == list(range(11))
    rows = np.array([[1, 2, 3, 1, 5], [4, 5, 6, 2, 3], [1, 2, 3, 7, 9]])
    assert dedup_weights(rows).tolist() == [0.0, 1.0, 1.0]                    # last (h,r,t) row wins


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    from rnnlogic_b200 import comm
    from rnnlogic_b200.trainer import allreduce_mean_grads, shard_indices
    comm.init_process_group("gloo", init_method="env://")
    torch.manual_seed(0)
    p = [torch.nn.Parameter(torch.zeros(5)), torch.nn.Parameter(torch.zeros(2, 3)), torch.nn.Parameter(torch.zeros(4))]
    p[0].grad = torch.full((5,), float(rank + 1))
    if rank == 1:
        p[1].grad = torch.ones(2, 3) * 4.0           # used by one rank only -> averaged with zeros
    allreduce_mean_grads(p, world)                    # p[2] unused everywhere -> stays None
    rows = torch.arange(5 * (rank + 2)).view(rank + 2, 5)
    cat = comm.cat_rows(rows)
    mine = shard_indices(9, world, rank)
    res = {"g0": p[0].grad.tolist(), "g1": p[1].grad.tolist(), "g2": p[2].grad, "cat": cat.shape[0], "mine": mine}
    torch.save(res, os.path.join(out, "r%d.pt" % rank))
    dist.barrier()
    dist.destroy_process_group()


def test_world2_gloo_collectives(tmp_path):
    import torch.multiprocessing as mp
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "r0.pt"), torch.load(tmp_path / "r1.pt")
    for r in (r0, r1):
        assert r["g0"] == [1.5] * 5 and r["g1"] == [[2.0] * 3] * 2 and r["g2"] is None and r["cat"] == 5
    assert len(r0["mine"]) == len(r1["mine"]) == 5 and set(r0["mine"]) | set(r1["mine"]) == set(range(9))


def test_compat_modules_resolve_the_reference_scripts_imports(monkeypatch, tmp_path):
    """`from data import ...`, `from predictors import ...`, ... of run_predictorplus.py / run_rnnlogic.py
    resolve through compat/ (names only; running them needs a GPU).  Generator-side names come from the
    reference's own files when its src/ follows compat/ on the path: a stand-in src/ that defines only
    those names takes its place here."""
    import importlib
    import sys
    compat = os.path.join(G.ROOT, "compat")
    monkeypatch.syspath_prepend(compat)
    for m in ("data", "predictors", "trainer", "comm", "utils", "_reference", "generators"):
        sys.modules.pop(m, None)
    wanted = {"data": ["KnowledgeGraph", "TrainDataset", "ValidDataset", "TestDataset"],
              "predictors": ["Predictor", "PredictorPlus"], "trainer": ["TrainerPredictor"],
              "utils": ["load_config", "save_config", "set_logger", "set_seed"], "comm": ["get_rank"]}
    for mod, names in wanted.items():
        module = importlib.import_module(mod)
        assert os.path.dirname(module.__file__) == compat
        for n in names:
            assert hasattr(module, n), (mod, n)
    import data
    with pytest.raises(AttributeError, match="outside the B200 hot path"):
        data.RuleDataset
    ref_src = tmp_path / "src"
    ref_src.mkdir()
    generator_side = {"data": ["RuleDataset", "Iterator"], "trainer": ["TrainerGenerator"], "generators": ["Generator"]}
    for mod, names in generator_side.items():
        (ref_src / (mod + ".py")).write_text("".join("class %s:\n    pass\n" % n for n in names))
    sys.path.append(str(ref_src))
    try:
        for mod, names in generator_side.items():
            module = importlib.import_module(mod)
            assert os.path.dirname(module.__file__) == compat
            for n in names:
                assert getattr(module, n).__module__ == "_reference_" + mod, (mod, n)
    finally:
        sys.path.remove(str(ref_src))
    for m in ("data", "predictors", "trainer", "comm", "utils", "_reference", "generators"):
        sys.modules.pop(m, None)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (CPU oracle port, no GPU needed) prints ONE JSON line with the keys the
    driver reads."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(G.ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3"],
                         capture_output=True, text=True, timeout=900, cwd=G.ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "rule_grounded_train_queries_per_sec" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_native_dataset_loader(tmp_path):
    """csrc_host/kg_loader.cpp == the reference's text parse (data.py:18-47,73-99): same ids, KeyError on
    an unknown name, names with spaces, blank lines and CRLF tolerated like line.strip()."""
    import time
    from rnnlogic_b200 import KnowledgeGraph
    fx = G.load("syn")
    N, R = int(fx["N"]), int(fx["R"])
    d = tmp_path / "ds"
    d.mkdir()
    (d / "entities.dict").write_text("".join("%d\tent %d\n" % (i, i) for i in range(N)))          # names with a space
    (d / "relations.dict").write_text("".join("%d\t!rel/%d\r\n" % (i, i) for i in range(R)))        # CRLF
    for split in ("train", "valid", "test"):
        body = "".join("ent %d\t!rel/%d\tent %d\n" % tuple(x) for x in fx[split].tolist())
        (d / (split + ".txt")).write_text(body + ("\n" if split == "valid" else ""))
    kg = KnowledgeGraph(str(d))
    assert kg.entity_size == N and kg.relation_size == R
    for split in ("train", "valid", "test"):
        assert np.array_equal(getattr(kg, split + "_array"), fx[split].astype(np.int64))
    assert kg.train_facts[0] == tuple(fx["train"][0].tolist()) and kg.entity2id["ent 3"] == 3
    (d / "test.txt").write_text("ent 1\t!rel/0\tnobody\n")
    with pytest.raises(KeyError):
        KnowledgeGraph(str(d))
    # FB15k-237-sized file: the parse itself takes a fraction of a second
    big = tmp_path / "big"
    big.mkdir()
    rng = np.random.default_rng(0)
    tri = np.stack([rng.integers(14541, size=544230), rng.integers(474, size=544230), rng.integers(14541, size=544230)], 1)
    (big / "entities.dict").write_text("".join("%d\t/m/%06d\n" % (i, i) for i in range(14541)))
    (big / "relations.dict").write_text("".join("%d\t/rel/%d\n" % (i, i) for i in range(474)))
    text = "".join("/m/%06d\t/rel/%d\t/m/%06d\n" % (h, r, t) for h, r, t in tri.tolist())
    (big / "train.txt").write_text(text)
    (big / "valid.txt").write_text("")
    (big / "test.txt").write_text("")
    from rnnlogic_b200.graph import _load_triples_native
    t0 = time.perf_counter()
    train, valid, test = _load_triples_native(str(big), 14541, 474)
    dt = time.perf_counter() - t0
    assert np.array_equal(train, tri) and valid.shape == (0, 3)
    assert dt < 5.0, dt


def test_binary_kg_cache(tmp_path, monkeypatch):
    """KnowledgeGraph(data_path, cache=dir): the second construction adopts the binary image (no parse, no
    sort) and is identical; touching a dataset file invalidates it; a read-only location is ignored."""
    from rnnlogic_b200 import KnowledgeGraph
    from rnnlogic_b200 import graph as graph_mod
    fx = G.load("syn")
    N, R = int(fx["N"]), int(fx["R"])
    d = tmp_path / "ds"
    d.mkdir()
    (d / "entities.dict").write_text("".join("%d\te%d\n" % (i, i) for i in range(N)))
    (d / "relations.dict").write_text("".join("%d\tr%d\n" % (i, i) for i in range(R)))
    for split in ("train", "valid", "test"):
        (d / (split + ".txt")).write_text("".join("e%d\tr%d\te%d\n" % tuple(x) for x in fx[split].tolist()))
    cache = tmp_path / "cache"
    a = KnowledgeGraph(str(d), cache=str(cache))
    files = list(cache.glob("kg_*.npz"))
    assert len(files) == 1
    calls = {"n": 0}
    real = graph_mod._load_triples_native
    monkeypatch.setattr(graph_mod, "_load_triples_native", lambda *x: (calls.__setitem__("n", calls["n"] + 1), real(*x))[1])
    monkeypatch.setattr(KnowledgeGraph, "_build_host", lambda self: (_ for _ in ()).throw(AssertionError("rebuilt")))
    b = KnowledgeGraph(str(d), cache=str(cache))                       # adopted: neither parsed nor rebuilt
    assert calls["n"] == 0
    for k in a.host:
        assert a.host[k].dtype == b.host[k].dtype and np.array_equal(a.host[k], b.host[k]), k
    for attr in ("train_array", "valid_array", "test_array", "train_edge_index", "rel_edges", "rel_rows", "rel_sources"):
        assert np.array_equal(getattr(a, attr), getattr(b, attr)), attr
    assert b.rank_words == a.rank_words and b.entity2id["e3"] == 3 and b.hr2o == a.hr2o
    assert np.array_equal(b.edge_index_of(fx["train"][:50]), a.edge_index_of(fx["train"][:50]))
    monkeypatch.undo()
    # one more train triple -> the key changes -> rebuilt and re-stored
    with open(d / "train.txt", "a") as f:
        f.write("e0\tr0\te%d\n" % (N - 1))
    c = KnowledgeGraph(str(d), cache=str(cache))
    assert c.train_array.shape[0] == a.train_array.shape[0] + 1
    # environment variable form
    monkeypatch.setenv("RNNLOGIC_B200_KG_CACHE", str(tmp_path / "cache2"))
    KnowledgeGraph(str(d))
    assert len(list((tmp_path / "cache2").glob("kg_*.npz"))) == 1


def test_step_prefetcher_order_errors_and_close():
    """data.StepPrefetcher: packed steps arrive in order from the loader thread, at most `depth` ahead; an
    exception in pack_fn surfaces in the consumer; close() releases a blocked producer."""
    import threading
    import time
    from rnnlogic_b200.data import StepPrefetcher
    seen = []

    def pack(x):
        seen.append(x)
        return x * 10

    pf = StepPrefetcher(pack, range(7), depth=2)
    time.sleep(0.3)
    assert len(seen) <= 3                                   # depth 2 in the queue + one being offered
    assert list(pf) == [0, 10, 20, 30, 40, 50, 60]

    def bad(x):
        if x == 2:
            raise KeyError("boom")
        return x

    pf = StepPrefetcher(bad, range(5), depth=1)
    assert next(pf) == 0 and next(pf) == 1
    with pytest.raises(KeyError):
        next(pf)
    pf = StepPrefetcher(lambda x: x, range(100), depth=1)
    assert next(pf) == 0
    pf.close()
    pf._thread.join(timeout=2.0)
    assert not pf._thread.is_alive()


def test_host_step_pack_layout():
    """engine.HostStep: the one-copy layout [h | t | arena_off | mask_off | item_off | int32: slot_head, q_off,
    nz_off, group_ptr] that Slots slices on the device; groups larger than 32 queries split into slots."""
    from rnnlogic_b200 import KnowledgeGraph, CompiledRules, parse_rules
    from rnnlogic_b200.engine import Grounder, HostStep
    fx = G.load("umls")
    kg = KnowledgeGraph(entity_size=int(fx["N"]), relation_size=int(fx["R"]), train=fx["train"])
    cr = CompiledRules(kg, parse_rules(G.rules_of(fx)))
    tri = fx["train"].astype(np.int64)
    batches = [tri[tri[:, 1] == q][:n] for q, n in ((3, 40), (5, 7), (3, 32), (8, 65)) if (tri[:, 1] == q).sum() >= n]
    assert len(batches) >= 3
    g = Grounder.__new__(Grounder)                     # pack_host touches no CUDA state
    g.cr = cr
    host = g.pack_host(batches, with_etr=True)
    sizes = [len(b) for b in batches]
    S = sum((n + 31) // 32 for n in sizes)
    Q = sum(sizes)
    assert (host.S, host.Q, host.k) == (S, Q, 2) and host.remove_query_edges and host.group_sizes == sizes
    pack = host.staged.numpy() if not host.staged.is_pinned() else host.staged.numpy()
    flat = np.concatenate(batches)
    assert np.array_equal(pack[:Q], flat[:, 0]) and np.array_equal(pack[Q:2 * Q], flat[:, 2])
    heads = np.concatenate([[int(b[0, 1])] * ((len(b) + 31) // 32) for b in batches])
    o = 2 * Q
    assert np.array_equal(pack[o:o + S], np.concatenate([[0], np.cumsum(cr.head_rows[heads])[:-1]]))
    assert np.array_equal(pack[o + S:o + 2 * S], np.concatenate([[0], np.cumsum(cr.head_chunks[heads])[:-1]]))
    assert np.array_equal(pack[o + 2 * S:o + 3 * S + 1], np.concatenate([[0], np.cumsum(cr.head_item_cap[heads])]))
    p32 = pack[host.n64:].view(np.int32)
    assert np.array_equal(p32[:S], heads)
    q_off = p32[S:2 * S + 1]
    assert q_off[0] == 0 and q_off[-1] == Q and (np.diff(q_off) <= 32).all() and (np.diff(q_off) > 0).all()
    gp = p32[3 * S + 1:3 * S + 1 + len(sizes) + 1]
    assert np.array_equal(np.diff(gp), [(n + 31) // 32 for n in sizes])
    assert host.nbytes == pack.nbytes and host.arena_rows == int(cr.head_rows[heads].sum())
    # single-slot groups carry no group table
    small = g.pack_host([b[:5] for b in batches], with_etr=False)
    assert small.ng1 == 0 and not small.remove_query_edges
    with pytest.raises(ValueError):
        Grounder._split([], [])


def test_snake_deal_partitions_and_balances():
    """trainer.snake_deal (bench.py's per-step dealing of batches to ranks): disjoint cover, equal counts,
    near-equal cost -- and identical to the largest-first snake order written out by hand."""
    from rnnlogic_b200.trainer import snake_deal
    rng = np.random.default_rng(4)
    for world in (1, 2, 4, 8):
        costs = (rng.pareto(1.2, size=64 * world) * 1000).astype(int).tolist()
        shares = [snake_deal(costs, world, r) for r in range(world)]
        flat = sorted(j for s in shares for j in s)
        assert flat == list(range(len(costs)))
        assert all(len(s) == 64 for s in shares)
        tot = [sum(costs[j] for j in s) for s in shares]
        assert max(tot) - min(tot) <= max(costs)                 # never further apart than one item
        order = sorted(range(len(costs)), key=lambda j: -costs[j])
        for r in range(world):
            want = [j for k, j in enumerate(order) if k % (2 * world) in (r, 2 * world - 1 - r)]
            assert shares[r] == want
    assert snake_deal([], 2, 0) == [] and snake_deal([5, 5, 5], 2, 0) == [0] and snake_deal([5, 5, 5], 2, 1) == [1, 2]


def test_launch_shape_feedback_host_logic():
    """Grounder.note_level_rows / chunks_per_warp (no CUDA needed): the density of a depth = non-zero rows the last calls
    produced per chunk of that depth; sparse frontiers keep long chunk runs per k_numeric warp, dense ones get short runs;
    dense mode and an unknown density fall back to the library default (0)."""
    import types
    import numpy as np
    from rnnlogic_b200.engine import Grounder
    gr = Grounder.__new__(Grounder)
    gr.force_dense, gr.level_density = False, {}
    gr.cr = types.SimpleNamespace(max_len=3, level_chunks=np.array([[100, 400, 300], [50, 200, 100]]))
    sl = types.SimpleNamespace(heads=np.array([0, 1, 1]))            # chunks per depth: 200, 800, 500
    assert [gr.chunks_per_warp(d) for d in (1, 2, 3)] == [0, 0, 0]
    gr.note_level_rows(sl, [0, 240, 4000, 4600, 0, 0, 0, 0])         # rows[d]: 1.2, 5.0, 9.2 per chunk
    assert [gr.chunks_per_warp(d) for d in (1, 2, 3)] == [16, 4, 1]
    gr.note_level_rows(sl, [0, 240, 5600, 2400, 0, 0, 0, 0])         # running mean with the previous call: 1.2, 6.0, 7.0
    assert abs(gr.level_density[2] - 6.0) < 1e-9 and [gr.chunks_per_warp(d) for d in (1, 2, 3)] == [16, 2, 2]
    gr.force_dense = True
    assert gr.chunks_per_warp(2) == 0
