"""Host-side driver of the grounding kernels: cuts a call's queries into 32-lane slots, owns the
frontier arena and runs the per-depth expansion launches (include/rnnlogic_b200.h).

Reference semantics: KnowledgeGraph.grounding / propagate (src/data.py:136-173) for every rule
of the batch's head relation at once."""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .rules import CompiledRules

LANES = _lib.LANES


def _stream():
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(torch.cuda.current_device()))


class HostStep:
    """The host half of a call: slot tables (and, for host batches, the queries) packed for ONE host->device
    copy.  Building it needs no CUDA work, so a loader thread can prepare steps ahead (data.StepPrefetcher)."""

    def __init__(self, cr: CompiledRules, heads: np.ndarray, q_off: np.ndarray, host_queries: Optional[np.ndarray] = None,
                 group_ptr: Optional[np.ndarray] = None, group_sizes=None, remove_query_edges: bool = False, pin: bool = True):
        S = int(heads.shape[0])
        self.S, self.heads, self.q_off = S, heads, q_off
        self.nq = np.diff(q_off)
        self.group_sizes = group_sizes
        self.remove_query_edges = bool(remove_query_edges)
        arena_off = np.zeros(S + 1, dtype=np.int64)
        np.cumsum(cr.head_rows[heads], out=arena_off[1:])
        nz_off = np.zeros(S + 1, dtype=np.int64)
        np.cumsum(cr.head_nodes[heads], out=nz_off[1:])
        mask_off = np.zeros(S + 1, dtype=np.int64)
        np.cumsum(cr.head_chunks[heads], out=mask_off[1:])
        item_off = np.zeros(S + 1, dtype=np.int64)
        np.cumsum(cr.head_item_cap[heads], out=item_off[1:])
        self.arena_rows, self.nz_total, self.mask_words = int(arena_off[-1]), int(nz_off[-1]), int(mask_off[-1])
        self.item_cap = int(item_off[-1])
        # int64 sections first, the int32 tables behind them
        self.k, self.Q = (0, 0) if host_queries is None else host_queries.shape
        self.ng1 = 0 if group_ptr is None else int(group_ptr.shape[0])
        k, Q, ng1 = self.k, self.Q, self.ng1
        self.n64 = n64 = k * Q + 3 * S + 1
        n32 = 3 * S + 1 + ng1
        pack = np.empty(n64 + (n32 + 1) // 2, dtype=np.int64)
        if k:
            pack[:k * Q] = host_queries.reshape(-1)
        o = k * Q
        pack[o:o + S] = arena_off[:-1]
        pack[o + S:o + 2 * S] = mask_off[:-1]
        pack[o + 2 * S:o + 3 * S + 1] = item_off
        p32 = pack[n64:].view(np.int32)
        p32[:S] = heads
        p32[S:2 * S + 1] = q_off
        p32[2 * S + 1:3 * S + 1] = nz_off[:-1]
        if ng1:
            p32[3 * S + 1:3 * S + 1 + ng1] = group_ptr
        self.nbytes = int(pack.nbytes)
        self.staged = torch.from_numpy(pack)
        if pin and torch.cuda.is_available():
            self.staged = self.staged.pin_memory()               # pinned staging for the async copy


class Slots:
    """Device-side description of one call (rl_slots) + its frontier arena."""

    def __init__(self, dg, host: HostStep, all_h: Optional[torch.Tensor] = None, all_t: Optional[torch.Tensor] = None,
                 etr: Optional[torch.Tensor] = None):
        """all_h / all_t / etr: int64 CUDA tensors -- or, when the HostStep carries the queries (rows h, t[, etr]),
        they travel with the slot descriptors in ONE pinned host->device copy."""
        dev = dg.device
        S, k, Q, ng1, n64 = host.S, host.k, host.Q, host.ng1, host.n64
        self.S, self.heads, self.q_off, self.nq = S, host.heads, host.q_off, host.nq
        self.arena_rows, self.nz_total, self.mask_words, self.item_cap = host.arena_rows, host.nz_total, host.mask_words, host.item_cap
        self.group_sizes = host.group_sizes
        d = host.staged.to(dev, non_blocking=True)
        self.h2d_bytes = host.nbytes
        if k:
            all_h, all_t = d[:Q], d[Q:2 * Q]
            etr = d[2 * Q:3 * Q] if k > 2 else None
        o = k * Q
        self.arena_off, self.mask_off, self.item_off = d[o:o + S], d[o + S:o + 2 * S], d[o + 2 * S:o + 3 * S + 1]
        d32 = d[n64:].view(torch.int32)
        self.slot_head, self.q_off_dev, self.nz_off = d32[:S], d32[S:2 * S + 1], d32[2 * S + 1:3 * S + 1]
        self.group_ptr_dev = d32[3 * S + 1:3 * S + 1 + ng1] if ng1 else None
        self.lane = torch.empty(4, S * LANES, dtype=torch.int32, device=dev)
        _lib.check(_lib.lib().rl_prepare_slots(
            dg.ref(), S, self.slot_head.data_ptr(), self.q_off_dev.data_ptr(), all_h.data_ptr(),
            all_t.data_ptr() if all_t is not None else None, etr.data_ptr() if etr is not None else None,
            int(host.remove_query_edges and etr is None),
            self.lane[0].data_ptr(), self.lane[1].data_ptr(), self.lane[2].data_ptr(), self.lane[3].data_ptr(),
            _stream()), "rl_prepare_slots")
        self.struct = _lib.RlSlots(S, self.slot_head.data_ptr(), self.lane[0].data_ptr(), self.lane[1].data_ptr(),
                                   self.lane[2].data_ptr(), self.lane[3].data_ptr(), self.arena_off.data_ptr(),
                                   self.nz_off.data_ptr(), self.mask_off.data_ptr())
        self._keep = (all_h, all_t, etr, d, host.staged)
        self.arena = None
        self.state = None         # int32 buffer: row_mask | node_cnt | item_cnt | bucket_cnt | overflow
        self.overflow = None
        self.frontier = None      # _lib.RlFrontier
        self.count_bits = 32

    def fref(self):
        return C.byref(self.frontier)

    def ref(self):
        return C.byref(self.struct)


class Grounder:
    """Grounds every rule of a compiled rule set for batches of queries on one device."""

    def __init__(self, graph, compiled: CompiledRules, device, force_dense: bool = False):
        self.graph, self.cr = graph, compiled
        self.dg = graph.device_graph(device)
        self.device = self.dg.device
        self.dr = compiled.device_rules(self.device)
        # a node takes ALL its rows (plain dense SpMM) once its parent has > dense_num/dense_den valid
        # rows; force_dense does so for every node (all algorithmic bytes of SURVEY 8d are moved)
        self.force_dense = bool(force_dense)
        self.dense_num, self.dense_den = 1, 4
        self.force_bits: Optional[int] = None
        self._ws_arena = None
        self._ws_state = None
        self._ws_items = None
        self._ws_cells = None
        self._ws_cells_cap = 0
        self.cell_cap = 0
        self.generation = 0           # bumped whenever a workspace is reallocated (captured CUDA graphs hold its pointers)
        self.level_density = {}       # depth -> non-zero rows per chunk seen by recent calls (see chunks_per_warp)
        self.level_events = None      # bench.py: list collecting (depth, start, end) CUDA events

    @staticmethod
    def _split(heads, sizes):
        """Cut single-relation groups into slots of <= 32 queries -> (slot heads, query offsets, group slot ranges)."""
        sh, qo, gp, pos = [], [0], [0], 0
        for hd, n in zip(heads, sizes):
            for k in range(0, int(n), LANES):
                sh.append(int(hd))
                qo.append(pos + min(int(n), k + LANES))
            pos += int(n)
            gp.append(len(sh))
        if not sh:
            raise ValueError("empty batch")
        return np.array(sh, dtype=np.int64), np.array(qo, dtype=np.int64), np.array(gp, dtype=np.int32), pos

    def make_slots(self, heads: Sequence[int], sizes: Sequence[int], all_h, all_t=None, etr=None,
                   coo_only: bool = False) -> Slots:
        """heads[i] / sizes[i]: head relation and number of queries of the i-th single-relation
        group; queries are consecutive in all_h / all_t / etr (int64 CUDA tensors).  Groups larger
        than 32 are split into several slots.  coo_only: the frontier is for the cell kernels (see make_slots_host)."""
        for name, t in (("all_h", all_h), ("all_t", all_t), ("edges_to_remove", etr)):
            if t is not None:
                _lib.require_cuda(t, name)
        sh, qo, gp, pos = self._split(heads, sizes)
        for name, t in (("all_h", all_h), ("all_t", all_t), ("edges_to_remove", etr)):
            if t is not None and int(t.numel()) != pos:
                raise ValueError("%s has %d entries for %d queries" % (name, int(t.numel()), pos))
        host = HostStep(self.cr, sh, qo, group_ptr=gp if len(sh) != len(sizes) else None, group_sizes=list(sizes))
        sl = Slots(self.dg, host, all_h.contiguous(), None if all_t is None else all_t.contiguous(),
                   None if etr is None else etr.contiguous())
        sl.coo_only = bool(coo_only)
        return sl

    def pack_host(self, batches, with_etr: bool, etr_lists=None) -> HostStep:
        """The CUDA-free half of make_slots_host (thread-safe: a loader thread may run it ahead of the step)."""
        if isinstance(batches[0], np.ndarray):                  # int arrays [n,3]: no per-triple Python work
            flat = np.concatenate(batches).astype(np.int64, copy=False).reshape(-1, 3)
            heads = [int(b[0, 1]) for b in batches]
        else:
            flat = np.array([x for b in batches for x in b], dtype=np.int64).reshape(-1, 3)
            heads = [b[0][1] for b in batches]
        sizes = [len(b) for b in batches]
        rows = [flat[:, 0], flat[:, 2]]
        if with_etr and etr_lists is not None:
            rows.append(np.array([e for l in etr_lists for e in l], dtype=np.int64))
        sh, qo, gp, pos = self._split(heads, sizes)
        return HostStep(self.cr, sh, qo, host_queries=np.stack(rows), group_ptr=gp if len(sh) != len(sizes) else None,
                        group_sizes=sizes, remove_query_edges=with_etr)

    def make_slots_host(self, batches, with_etr: bool, etr_lists=None, coo_only: bool = False) -> Slots:
        """Slots for a list of single-relation batches given as host lists of (h, r, t) triples
        (what the datasets hold) -- or for a HostStep packed ahead by pack_host.  ONE packed host->device copy
        carries h, t and the slot tables.  with_etr: every query's own train edge is masked out
        (data.py:214-216); the edge is found on the device unless etr_lists gives the reference's
        per-relation edge indices explicitly."""
        host = batches if isinstance(batches, HostStep) else self.pack_host(batches, with_etr, etr_lists)
        sl = Slots(self.dg, host)
        sl.use_workspace = True
        sl.coo_only = bool(coo_only)      # cell paths walk the items as appended: no entity-grouped copy, no bucket tables
        return sl

    def _layout(self, sl: "Slots | HostStep", bits: int = 32):
        """Sizes (in int32 words) of the three per-call buffers: arena | zeroed state | scratch."""
        W, N, S = self.graph.rank_words, self.graph.entity_size, sl.S
        n_mask, n_cnt = sl.mask_words + 1, sl.nz_total + 1
        n_bkt = S * (W * 32 + 32)                                        # per-entity item counts / offsets (RL_BUCKET_STRIDE)
        n_pad = -(n_mask + n_cnt + S) % 4                                # the bucket table is read with 16-byte loads
        cap = max(1, sl.item_cap)
        o_nz = n_mask + n_cnt + S + n_pad + n_bkt
        o_sc = 10 * cap + n_bkt
        return {
            "arena": max(1, sl.arena_rows) * LANES * (1 if bits == 32 else 2),
            # zeroed: row bitmaps | node counts | item counts | pad | buckets | candidate words | cell counters[8] | overflow | rows per depth[8]
            "o_cnt": n_mask, "o_icnt": n_mask + n_cnt, "o_bkt": n_mask + n_cnt + S + n_pad,
            "o_nz": o_nz, "o_ctr": o_nz + S * N, "state": o_nz + S * N + 8 + 1 + 8,
            # scratch: items | items_sorted (int32x4 records, exact upper bound) | bucket offsets | item lane masks (x2) |
            # first cell per (slot, entity) | cells per slot | per-query CE statistics (x2)
            "n_items": 4 * cap, "o_boff": 8 * cap, "o_im": 8 * cap + n_bkt, "o_ims": 9 * cap + n_bkt,
            "o_coff": o_sc, "o_ncell": o_sc + S * N, "o_qmax": o_sc + S * N + S, "o_qsum": o_sc + S * N + S + S * LANES,
            "scratch": o_sc + S * N + S + 2 * S * LANES,
        }

    def _run(self, sl: Slots, bits: int):
        dev = self.device
        sl.count_bits = bits
        lay = self._layout(sl, bits)
        n_arena, n_state, n_scratch = lay["arena"], lay["state"], lay["scratch"]
        if getattr(sl, "use_workspace", False):
            # fused paths consume the frontier inside the call: reuse grow-only buffers (no cudaMalloc in
            # steady state; the arena needs no clearing, rows outside the bitmap are never read)
            if self._ws_arena is None or self._ws_arena.numel() < n_arena:
                self._ws_arena = None
                self._ws_arena = torch.empty(int(n_arena * 1.25), dtype=torch.int32, device=dev)
                self.generation += 1
            if self._ws_state is None or self._ws_state.numel() < n_state:
                self._ws_state = torch.empty(int(n_state * 1.25), dtype=torch.int32, device=dev)
                self.generation += 1
            if self._ws_items is None or self._ws_items.numel() < n_scratch:
                self._ws_items = None
                self._ws_items = torch.empty(int(n_scratch * 1.25), dtype=torch.int32, device=dev)
                self.generation += 1
            sl.arena = self._ws_arena[:n_arena]
            sl.state = self._ws_state[:n_state].zero_()
            scratch = self._ws_items[:n_scratch]
        else:
            sl.arena = torch.empty(n_arena, dtype=torch.int32, device=dev)
            sl.state = torch.zeros(n_state, dtype=torch.int32, device=dev)                    # one memset
            scratch = torch.empty(n_scratch, dtype=torch.int32, device=dev)
        sl.scratch = scratch
        sl.overflow = sl.state[lay["o_ctr"] + 8:lay["o_ctr"] + 9]
        sl.cell_counters = sl.state[lay["o_ctr"]:lay["o_ctr"] + 8]
        sl.slot_ncell = scratch[lay["o_ncell"]:lay["o_ncell"] + sl.S]
        sl.flags = sl.state[lay["o_ctr"]:]                 # cell counters[8] | count overflow | non-zero rows per depth[8]: one D2H read
        sl.nzmask = sl.state[lay["o_nz"]:lay["o_ctr"]].view(sl.S, -1)     # candidate word of every (slot, entity)
        base, sb = sl.state.data_ptr(), scratch.data_ptr()
        coo_only = bool(getattr(sl, "coo_only", False))                  # cell paths: no entity-grouped copy of the items
        sl.frontier = _lib.RlFrontier(bits, sl.arena.data_ptr(), base, base + 4 * lay["o_cnt"],
                                      sl.overflow.data_ptr(), sb, sb + 4 * lay["n_items"], sl.item_off.data_ptr(),
                                      base + 4 * lay["o_icnt"], None if coo_only else base + 4 * lay["o_bkt"],
                                      sb + 4 * lay["o_boff"], sb + 4 * lay["o_im"], sb + 4 * lay["o_ims"], base + 4 * lay["o_nz"])
        sl.cells_tables = {"counters": base + 4 * lay["o_ctr"], "nzmask": base + 4 * lay["o_nz"], "cand_off": sb + 4 * lay["o_coff"],
                           "slot_ncell": sb + 4 * lay["o_ncell"], "qmax": sb + 4 * lay["o_qmax"], "qsum": sb + 4 * lay["o_qsum"]}
        sl.cells = None
        L = _lib.lib()
        lc = self.cr.level_chunks[sl.heads]                               # [S, max_len]
        ln = self.cr.level_sym_items[sl.heads]
        for depth in range(1, self.cr.max_len + 1):
            gc, gn = int(lc[:, depth - 1].max()), int(ln[:, depth - 1].max())
            if gc == 0:
                continue
            if self.level_events is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            _lib.check(L.rl_expand_level(self.dg.ref(), self.dr.ref(), sl.ref(), depth, gn, gc, sl.fref(),
                                         self.dense_num, self.dense_den, int(self.force_dense), self.chunks_per_warp(depth), _stream()),
                       "rl_expand_level")
            if self.level_events is not None:
                e1.record()
                self.level_events.append((depth, e0, e1))

    # ---- launch-shape feedback -------------------------------------------------------------------
    # k_numeric gives one warp a run of consecutive 32-row chunks.  Long runs win when most chunks are empty (i.i.d.
    # graphs: ~1 non-zero row per chunk), short runs when the frontier stays alive (typed graphs: ~9 rows per chunk; a
    # 16-chunk run is then a warp's worth of thousands of entries and the launch ends on a few stragglers).  The kernel
    # counts the non-zero rows it produced per depth (rl_frontier.overflow[1 + d]); whoever reads a call's flags back
    # hands them to note_level_rows and the NEXT call is launched with the run length that density asks for
    # (swept on the B200: profiles/README.md).
    def chunks_per_warp(self, depth: int) -> int:
        d = self.level_density.get(depth)
        if self.force_dense or d is None:
            return 0                                                     # library default
        return 16 if d < 4.0 else 4 if d < 6.0 else 2 if d < 8.0 else 1      # measured: i.i.d. 1.2 -> 16, WN18RR shape ~3 -> 16, typed 6-9 -> 2 / 1

    def note_level_rows(self, sl, rows) -> None:
        """rows[d] = non-zero rows the call produced at depth d (flags[9:17] of the call)."""
        lc = self.cr.level_chunks[sl.heads]
        for depth in range(1, min(self.cr.max_len, 7) + 1):
            chunks = float(lc[:, depth - 1].sum())
            if chunks > 0:
                dens = float(rows[depth]) / chunks
                old = self.level_density.get(depth)
                self.level_density[depth] = dens if old is None else 0.5 * (old + dens)

    # ---- candidate cells (rl_cells) ------------------------------------------------------------
    cells_per_slot_hint = 24576       # first guess of the per-cell capacity; grows on demand (see ensure_cell_cap)

    def cell_capacity(self, sl: Slots) -> int:
        """Cells the per-cell arrays of a call are sized for: the largest count seen so far or the per-slot hint."""
        return (max(self.cell_cap, self.cells_per_slot_hint * sl.S) + 63) // 64 * 64       # planes stay 16-byte aligned

    def cell_arrays(self, sl: Slots, planes: int):
        """Grow-only per-cell workspace of ``planes`` 32-bit planes [cap] each -> (cap, flat fp32 tensor)."""
        want = self.cell_capacity(sl)
        n = want * planes
        if self._ws_cells is None or self._ws_cells.numel() < n or self._ws_cells_cap < want:
            self._ws_cells = None
            self._ws_cells = torch.empty(n, dtype=torch.float32, device=self.device)
            self._ws_cells_cap = want
            self.generation += 1
        return self._ws_cells_cap, self._ws_cells

    def build_cells(self, sl: Slots, floats_per_cell: int, cap: Optional[int] = None):
        """rl_cells_build for an expanded frontier -> (RlCells, fp32 planes [floats_per_cell][cap]).
        cap=None: the arrays live in the grounder's grow-only workspace, which the next call reuses (fused steps
        consume them within the call).  Else fresh arrays for ``cap`` cells that belong to ``sl`` alone."""
        if cap is None:
            cap, ws = self.cell_arrays(sl, 2 + floats_per_cell)
        else:
            cap = (max(1, int(cap)) + 63) // 64 * 64
            ws = torch.empty(cap * (2 + floats_per_cell), dtype=torch.float32, device=self.device)
        sl.cell_ws = ws                                                   # keeps the arrays alive as long as the call
        keys, ents = ws[:cap].view(torch.int32), ws[cap:2 * cap]          # plane 1: the cells' entities
        t = sl.cells_tables
        sl.cells = _lib.RlCells(cap, t["counters"], t["nzmask"], t["cand_off"], keys.data_ptr(), ents.data_ptr(),
                                t["slot_ncell"], t["qmax"], t["qsum"])
        sl.cell_cap = cap
        _lib.check(_lib.lib().rl_cells_build(self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), C.byref(sl.cells), _stream()),
                   "rl_cells_build")
        return sl.cells, ws[2 * cap:(2 + floats_per_cell) * cap].view(floats_per_cell, cap)

    def note_cell_count(self, n_cells: int):
        """Remember the largest cell count seen so that later calls size their arrays for it (x1.25)."""
        self.cell_cap = max(self.cell_cap, int(n_cells * 1.25) + 1024)

    def reserve(self, slots_list):
        """Size the reusable frontier workspace for the largest of the given calls up front, so that no
        step of a steady-state loop triggers a cudaMalloc."""
        lays = [self._layout(sl) for sl in slots_list]
        for name, key in (("_ws_arena", "arena"), ("_ws_state", "state"), ("_ws_items", "scratch")):
            n = max(l[key] for l in lays)
            cur = getattr(self, name)
            if cur is None or cur.numel() < n:
                setattr(self, name, None)
                setattr(self, name, torch.empty(n, dtype=torch.int32, device=self.device))
                self.generation += 1

    def reserve_single_slot(self):
        """Size the frontier workspace for one slot of the LARGEST head, so that per-head CUDA graphs of the reference
        schedule (one batch per step) never see a reallocation."""
        cr = self.cr
        if not len(cr.head_rows):
            return

        class _One:                                              # what _layout reads of a call
            S = 1
        one = _One()
        one.arena_rows, one.nz_total = int(cr.head_rows.max()), int(cr.head_nodes.max())
        one.mask_words, one.item_cap = int(cr.head_chunks.max()), int(cr.head_item_cap.max())
        lay = self._layout(one)
        for name, key in (("_ws_arena", "arena"), ("_ws_state", "state"), ("_ws_items", "scratch")):
            cur = getattr(self, name)
            if cur is None or cur.numel() < lay[key]:
                setattr(self, name, None)
                setattr(self, name, torch.empty(lay[key], dtype=torch.int32, device=self.device))
                self.generation += 1

    def _run_empty(self, sl: Slots):
        sl.arena = torch.zeros(LANES, dtype=torch.int32, device=self.device)
        sl.state = torch.zeros(8, dtype=torch.int32, device=self.device)
        sl.overflow = sl.state[-1:]
        p = sl.state.data_ptr()
        sl.frontier = _lib.RlFrontier(32, sl.arena.data_ptr(), p, p + 4, sl.overflow.data_ptr(),
                                      None, None, None, None, None, None, None, None, None)

    def ground(self, sl: Slots, check_overflow: bool = True) -> Slots:
        """Run all depths.  Counts are kept in 32-bit rows; if any count does not fit (host sync on
        one int when check_overflow) the call is repeated with 64-bit rows, which wrap exactly
        like the reference's int64 tensors."""
        bits = self.force_bits or 32
        self._run(sl, bits)
        if bits == 32 and check_overflow and int(sl.overflow.item()) != 0:
            self._run(sl, 64)
        return sl

    def node_counts(self, sl: Slots, slot: int, node: int) -> torch.Tensor:
        """int64[32, N] dense counts of one trie node (node < 0: the one-hot root)."""
        out = torch.empty(LANES, self.graph.entity_size, dtype=torch.int64, device=self.device)
        if sl.frontier is None:                       # only the one-hot root is asked for (empty body)
            self._run_empty(sl)
        _lib.check(_lib.lib().rl_node_counts_dense(
            self.dg.ref(), self.dr.ref(), sl.ref(), slot, node, sl.fref(), out.data_ptr(), _stream()),
            "rl_node_counts_dense")
        return out

    def rule_counts(self, sl: Slots, rule_ids: Sequence[int]) -> torch.Tensor:
        """int64[len(rule_ids), Q, N] counts per rule (debug / parity; the production path never
        materialises this tensor).  All slots must share the rules' head."""
        Q = int(sl.q_off[-1])
        out = torch.empty(len(rule_ids), Q, self.graph.entity_size, dtype=torch.int64, device=self.device)
        for i, rid in enumerate(rule_ids):
            node = int(self.cr.rule_node[rid])
            for s in range(sl.S):
                dense = self.node_counts(sl, s, node)
                out[i, sl.q_off[s]:sl.q_off[s + 1]] = dense[:sl.nq[s]]
        return out


_CHAIN_CACHE_MAX = 4096


def ground_chain(graph, h: torch.Tensor, r: int, body: List[int], etr: Optional[torch.Tensor]) -> torch.Tensor:
    """KnowledgeGraph.grounding for one rule body (src/data.py:136-147)."""
    _lib.require_cuda(h, "h")
    key = (r, tuple(body))
    cache = graph._chains
    if key in cache:
        cache.move_to_end(key)
        cr = cache[key]
    else:
        cr = CompiledRules(graph, [(r, body)])
        cache[key] = cr
        if len(cache) > _CHAIN_CACHE_MAX:
            cache.popitem(last=False)
    grs = cr.__dict__.setdefault("_grounders", {})               # one driver (and workspace) per cached chain and device
    gr = grs.get(str(h.device))
    if gr is None:
        gr = grs[str(h.device)] = Grounder(graph, cr, h.device)
    B = int(h.shape[0])
    sl = gr.make_slots([r], [B], h.to(torch.int64), None, None if etr is None else etr.to(h.device, torch.int64))
    if len(body):
        gr.ground(sl)
    return gr.rule_counts(sl, [0])[0]
