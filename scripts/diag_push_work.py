"""Work of the frontier expansion per trie depth, pull against push, on the bench workload (i.i.d. or --typed graph).
Grounds sample batches of the headline step and counts, from the expanded frontier:
  rows     valid (non-zero) destination rows
  scanned  pair-table entries the pull scans for them (depth 1: in-edges of the row)
  pairs    live (parent row, out-edge) pairs: what a push formulation walks (and what the pull fetches)
  cells    non-zero (pair, lane) cells: the atomics a push issues
  lanes    depth 1: non-zero lanes per valid row (a search per (row, lane) finds nothing for the others)
usage: python scripts/diag_push_work.py [--typed] [--batches 32]"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--typed", action="store_true")
    ap.add_argument("--batches", type=int, default=32)
    a = ap.parse_args()
    from rnnlogic_b200 import KnowledgeGraph, CompiledRules
    from rnnlogic_b200.engine import Grounder
    shape, N, R, train, valid, test, rules = bench.build_workload("fb15k237", typed=a.typed)
    batches = bench.make_batches(train, R, seed=1)[:a.batches]
    kg = KnowledgeGraph(entity_size=N, relation_size=R, train=train, valid=valid, test=test)
    cr = CompiledRules(kg, rules)
    gr = Grounder(kg, cr, torch.device("cuda:0"))
    sl = gr.make_slots_host(batches, with_etr=True)
    sl.use_workspace = False
    gr.force_bits = 64
    gr.ground(sl)
    arena = sl.arena.view(torch.int64).cpu().numpy().reshape(-1, 32)
    nzl = (arena != 0).sum(1)
    masks = sl.state[:sl.mask_words].cpu().numpy().view(np.uint32)
    arena_off, mask_off = sl.arena_off.cpu().numpy(), sl.mask_off.cpu().numpy()
    h = kg.host
    dst_ptr, row_dst, row_start = h["dst_ptr"].astype(np.int64), h["row_dst"], h["row_start"].astype(np.int64)
    outdeg = np.zeros((R, N), dtype=np.int64)                    # out-edges of entity e under relation r
    np.add.at(outdeg, (train[:, 1], train[:, 0]), 1)
    pair_ptr = gr.dr.t["pair_ptr"].cpu().numpy().astype(np.int64)
    rec = cr.host["node_rec"].reshape(-1, 8)
    row_off, prow_off, pair_off = cr.host["node_row_off"], cr.host["node_prow_off"], cr.host["node_pair_off"]
    lvl = cr.host["lvl_ptr"].reshape(R, -1)
    L = cr.max_len
    rows, scanned, pairs, cells = (np.zeros(L + 1, np.int64) for _ in range(4))
    lanes1 = []

    def valid_rows(s, q, v):
        D, c0 = int(rec[v, 4]), int(rec[v, 5])
        m = masks[mask_off[s] + c0 - lvl[q, 0]: mask_off[s] + c0 - lvl[q, 0] + (D + 31) // 32]
        bits = np.unpackbits(m.view(np.uint8), bitorder="little")[:D]
        return np.flatnonzero(bits)

    for s, q in enumerate(sl.heads):
        for v in range(int(cr.head_node_ptr[q]), int(cr.head_node_ptr[q + 1])):
            d = int(cr.node_depth[v])
            rho, p, prel, gbase = (int(x) for x in rec[v, :4])
            vr = valid_rows(s, q, v)
            rows[d] += vr.size
            if d == 1:
                scanned[d] += int((row_start[gbase + vr + 1] - row_start[gbase + vr]).sum())
                lanes1.append(nzl[arena_off[s] + row_off[v] + vr])
                pairs[d] += int(nzl[arena_off[s] + row_off[v] + vr].sum())       # one add per (query, edge) ...
                cells[d] += int(arena[arena_off[s] + row_off[v] + vr].sum())     # ... counted with multiplicity
                continue
            if vr.size:
                scanned[d] += int((pair_ptr[pair_off[v] + vr + 1] - pair_ptr[pair_off[v] + vr]).sum())
            pr = valid_rows(s, q, p)
            if pr.size:
                deg = outdeg[rho, row_dst[dst_ptr[prel] + pr]]
                pairs[d] += int(deg.sum())
                cells[d] += int((deg * nzl[arena_off[s] + prow_off[v] + pr]).sum())
    print("%s graph, %d batches (%d slots)" % ("typed" if a.typed else "i.i.d.", len(batches), sl.S))
    print("depth %10s %12s %12s %12s" % ("rows", "scanned", "pairs", "cells"))
    for d in range(1, L + 1):
        if rows[d]:
            print("%5d %10d %12d %12d %12d" % (d, rows[d], scanned[d], pairs[d], cells[d]))
    l1 = np.concatenate(lanes1) if lanes1 else np.zeros(1)
    print("depth 1: non-zero lanes per valid row: mean %.2f, median %d, max %d (of 32)"
          % (l1.mean(), int(np.median(l1)), int(l1.max())))


if __name__ == "__main__":
    main()
