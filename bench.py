#!/usr/bin/env python
"""bench.py -- rule-grounded queries/sec on the FB15k-237-shaped synthetic workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path (ground every rule of the head -> candidate cells -> rule-weight aggregation ->
log(softmax+1e-8) CE -> backward into rule weights/bias -> Adam) over ``--batches`` reference batches
(single-relation groups of <= 32 train queries, src/data.py:186-196) per GPU.  Batches are sharded over ranks
(KG + rules replicated, one flat gradient all-reduce per step): weak scaling.  ``value`` is timed with the
step's queries already in HBM; ``e2e`` goes through the public fused API from HOST arrays (pack + H2D + kernels +
D2H of the losses) every step.  ``configs`` holds the same end-to-end measurement for the other configurations
BASELINE.json names (PredictorPlus as shipped for FB15k-237, with a RotatE-shaped entity feature, the WN18RR
config), for a TYPED synthetic graph whose rule bodies compose, and for the reference's own schedule (one
32-query batch per optimizer step).  ``--impl reference`` times the CPU oracle port of the reference path."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rule_grounded_train_queries_per_sec"
UNIT = "queries/s"
B = 32


def build_workload(name="fb15k237", typed=False):
    from rnnlogic_b200 import synth
    shape = synth.load_shape(name)
    if typed:
        N, R, train, valid, test, meta = synth.typed_kg(shape)
        rules = synth.typed_rules(shape, meta)
    else:
        N, R, train, valid, test = synth.synthetic_kg(shape)
        rules = synth.synthetic_rules(shape)
    return shape, N, R, train, valid, test, rules


def make_batches(train, R, seed):
    """Reference batching (data.py:186-196) with numpy: group by relation, shuffle, cut into <= 32."""
    rng = np.random.default_rng(seed)
    batches = []
    order = np.argsort(train[:, 1], kind="stable")
    tr = train[order]
    bounds = np.searchsorted(tr[:, 1], np.arange(R + 1))
    for r in range(R):
        grp = tr[bounds[r]:bounds[r + 1]]
        grp = grp[rng.permutation(grp.shape[0])]
        for k in range(0, grp.shape[0], B):
            batches.append(grp[k:k + B])
    perm = rng.permutation(len(batches))
    return [batches[i] for i in perm]


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_run(N, R, train, valid, test, rules, batches, steps, warmup, per, sample=8, budget_s=20.0):
    """Oracle port of the reference Predictor train step on host cores.  A step of the GPU arm is ``per`` batches with
    one optimizer step; the CPU arm times a BOUNDED SAMPLE of such a step: ``sample`` of its batches (gradients of
    loss / per accumulated) and the optimizer step."""
    from oracle import rnnlogic_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    kg = O.OracleKG(N, R, train, valid, test)
    table = O.relation2rules(O.parse_rules([[h] + list(b) for h, b in rules]), R)
    g = torch.Generator().manual_seed(0)
    w = (torch.randn(len(rules), generator=g) * 0.1).requires_grad_()
    bias = torch.zeros(N, requires_grad=True)
    opt = torch.optim.Adam([w, bias], lr=0.005)
    sample = max(1, min(sample, per))
    times, nq = [], 0
    cursor = [0]

    def one_step():
        opt.zero_grad()
        q_done = 0
        for _ in range(sample):
            batch = batches[cursor[0] % len(batches)]
            cursor[0] += 1
            data = [tuple(int(v) for v in row) for row in batch]
            all_h, all_r, all_t, target, etr = O.train_batch(kg, data)
            q = int(all_r[0])
            score, mask = O.predictor_forward(kg, table[q], w, bias, all_h, etr.numpy(), q)
            loss = O.ce_loss(score, mask, O.smoothed_target(target, all_t, 0.2))
            (loss / per).backward()
            q_done += len(data)
        opt.step()
        return q_done

    for _ in range(warmup):
        one_step()
    t_all = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        nq += one_step()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s and len(times) >= 1:
            break
    total = sum(times)
    return {"value": nq / total, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d steps, each %d of the step's %d train batches of <=32 queries (%d queries in all) + the optimizer "
                      "step; oracle port: C grounding per rule (1 thread) + torch-CPU aggregation/CE/backward/Adam (%d threads)"
                      % (len(times), sample, per, nq, torch.get_num_threads()),
            "steps_done": len(times), "ms_per_step": 1e3 * total / len(times)}


class quiet_gc:
    """Timed regions run with the long-lived objects FROZEN out of the cyclic garbage collector's generations: the rule set
    alone is ~10^6 small Python objects, and a generation-2 pass over them in the middle of a loop is a 30-70 ms host stall
    that drains the GPU queue (and, through the per-step all-reduce, stalls every other rank too).  The collector itself
    stays on -- PredictorPlus steps create cyclic garbage that holds device memory -- it just has nothing old to walk."""

    def __init__(self, model=None):
        # Predictor loops only: with PredictorPlus (autograd through the rule encoder) runs with frozen generations were
        # bimodal on the B200 (4.06 vs 6.7 ms per step, 3 of 5 runs slow; 0 of 8 with the collector untouched)
        self.plain = model is None or type(model).__name__ == "Predictor"

    def __enter__(self):
        import gc
        self.on = self.plain and os.environ.get("RL_BENCH_KEEP_GC") is None      # A/B switch
        if self.on:
            gc.collect()
            gc.freeze()

    def __exit__(self, *exc):
        import gc
        if self.on:
            gc.unfreeze()


class Runner:
    """One model + optimizer on this rank with its dealt steps: device-resident and end-to-end loops."""
    read_late = 2        # e2e: a step's losses are read this many steps behind the enqueue front (absorbs host jitter)

    def __init__(self, model, step_lists, per, world, dev, lr=0.005):
        from rnnlogic_b200.optim import Adam
        from rnnlogic_b200 import cellpath
        self.model, self.steps, self.per, self.world, self.dev = model, step_lists, per, world, dev
        self.cellpath = cellpath
        self.params = model.fused_params()
        self.opt = Adam(self.params, lr=lr)          # torch.optim.Adam semantics, one element per thread (rl_adam_step)
        self.sk = model._driver(dev)
        self.queries = [sum(len(b) for b in sb) for sb in step_lists]

    def start_allreduce(self, gbuf):
        if self.world == 1:
            return None
        return torch.distributed.all_reduce(gbuf.flat, op=torch.distributed.ReduceOp.SUM, async_op=True)

    def finish_step(self, work, gbuf):
        if work is not None:
            work.wait()
            gbuf.flat.div_(self.world)
        gbuf.assign()
        self.opt.step()

    def size_cells(self):
        """One synchronous pass over the distinct steps so that the per-cell arrays fit every step (no overflow and
        no cudaMalloc inside a timed loop)."""
        from rnnlogic_b200.predictors import RlStepOverflow
        for sb in self.steps:
            for _ in range(3):
                tk = self.model.submit_train_step(sb, 0.2, grad_scale=1.0 / self.per)
                try:
                    tk.result()
                    break
                except RlStepOverflow as e:
                    if tk.count_overflow:
                        raise AssertionError("32-bit count overflow on the bench workload: " + str(e))
        torch.cuda.synchronize()

    def _device_loop(self, warmup, steps, level_events=False):
        """Queries already in HBM.  -> (ms, queries, launches, flags, level events)."""
        from rnnlogic_b200 import _lib
        model, sk, per = self.model, self.sk, self.per
        n_steps = warmup + steps
        slots = [sk.gr.make_slots_host(self.steps[s % len(self.steps)], with_etr=True, coo_only=not getattr(self, 'dense_tail', False)) for s in range(n_steps)]
        sk.gr.reserve(slots)
        self.slots = slots
        torch.cuda.synchronize()
        if self.world > 1:
            torch.distributed.barrier()
        flags_acc = torch.zeros(17, dtype=torch.int32, device=self.dev)
        for s in range(warmup):
            gbuf = self.cellpath.GradBuffer(self.params)
            model.step_on_slots(sk, slots[s], 0.2, 1.0 / per, gbuf)
            flags_acc += slots[s].flags                  # (also warms the op: its first call loads a module, ~17 ms)
            sk.gr.note_level_rows(slots[s], slots[s].flags[9:17].tolist())     # warm-up only: launch-shape feedback (a host read)
            self.finish_step(self.start_allreduce(gbuf), gbuf)
        flags_acc.zero_()
        torch.cuda.synchronize()
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        launches0 = _lib.lib().rl_launch_count()
        sk.gr.level_events = [] if level_events else None
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        losses = []
        sk.gr._run(slots[warmup], 32)
        dbg = os.environ.get("RL_BENCH_TRACE")
        step_ev = []
        for s in range(warmup, n_steps):
            if dbg:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                step_ev.append(ev)
            t0 = time.perf_counter()
            gbuf = self.cellpath.GradBuffer(self.params)
            t1 = time.perf_counter()
            loss, tsum = model.step_on_slots(sk, slots[s], 0.2, 1.0 / per, gbuf, expanded=True)
            t2 = time.perf_counter()
            flags_acc += slots[s].flags                  # the workspace is reused by the next step
            t2b = time.perf_counter()
            pending = self.start_allreduce(gbuf)
            if s + 1 < n_steps:                          # grounding is parameter-independent: enqueue it before the exchange
                sk.gr._run(slots[s + 1], 32)
            t3 = time.perf_counter()
            if dbg and s < warmup + 3:
                print("[trace] flags %.2f ms" % ((t2b - t2) * 1e3), file=sys.stderr)
            self.finish_step(pending, gbuf)
            losses.append(loss)
            if dbg and s < warmup + 6:
                print("[trace] gbuf %.2f step %.2f run %.2f finish %.2f ms" % ((t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3,
                                                                              (time.perf_counter() - t3) * 1e3), file=sys.stderr)
        ev1.record()
        torch.cuda.synchronize()
        if self.world > 1:
            torch.distributed.barrier()
        self.last_step = (loss, tsum, gbuf)
        ms = ev0.elapsed_time(ev1)
        if dbg and len(step_ev) > 1:
            per = [step_ev[i].elapsed_time(step_ev[i + 1]) for i in range(len(step_ev) - 1)]
            print("[trace] device ms per step: " + " ".join("%.2f" % v for v in per), file=sys.stderr)
        launches = _lib.lib().rl_launch_count() - launches0
        events, sk.gr.level_events = sk.gr.level_events, None
        flags = flags_acc.cpu().numpy()
        assert flags[8] == 0, "32-bit count overflow inside the timed region"
        assert flags[1] == 0, "cell arrays overflowed inside the timed region"
        assert all(torch.isfinite(l).all().item() for l in losses)
        return ms, sum(self.queries[s % len(self.steps)] for s in range(warmup, n_steps)), launches, events

    def _graph_loop(self, warmup, steps):
        """The reference's schedule (one batch per optimizer step) through the per-head CUDA graphs, the way
        TrainerPredictor.train drives them: host arrays in, loss out; per step two graph replays (grounding of step k+1
        enqueued behind the scoring of step k), one event wait, one optimizer step.  -> (ms, queries)"""
        from rnnlogic_b200 import cellpath
        from rnnlogic_b200.predictors import _used_params
        model = self.model
        seq = [np.asarray(self.steps[s % len(self.steps)][0], dtype=np.int64).reshape(-1, 3) for s in range(warmup + steps)]
        for b in seq:                                            # capture the graphs of the heads of this run (one each)
            cellpath.graph_train_step(model, b, 0.2)
        torch.cuda.synchronize()
        if self.world > 1:
            torch.distributed.barrier()
        nq = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gs_next = None
        for s, b in enumerate(seq):
            if s == warmup:
                e0.record()
            gs, gs_next = gs_next, None
            if gs is None:
                gs = cellpath.graph_step_for(model, b, 0.2)
                gs.launch_ground(b)
            gs.launch_score()
            if s + 1 < len(seq):
                gs_next = cellpath.graph_step_for(model, seq[s + 1], 0.2)
                gs_next.launch_ground(seq[s + 1])
            res = cellpath.graph_step_result(model, gs)
            assert res is not None and np.isfinite(res[0]), "a bench batch needed the eager path (count overflow / cell arrays)"
            if self.world > 1:                                   # the path's one collective: the flat gradient buffer of the graph
                torch.distributed.all_reduce(res[3].flat, op=torch.distributed.ReduceOp.SUM)
                res[3].flat.div_(self.world)
            res[3].assign(_used_params(model, res[2]))
            self.opt.step()
            if s >= warmup:
                nq += len(b)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), nq

    def _e2e_loop(self, warmup, steps, trace=None):
        """Host int arrays in, losses out, through submit / prepare / finish / result (software-pipelined: a
        step's losses are read ``read_late`` steps behind the enqueue front; every step does its own packed H2D copy and its
        own D2H read inside the timed region).  -> (ms, queries, h2d, d2h)."""
        from rnnlogic_b200.data import StepPrefetcher
        model, per = self.model, self.per
        n_steps = warmup + steps
        seq = [self.steps[s % len(self.steps)] for s in range(n_steps)]
        torch.cuda.synchronize()
        if self.world > 1:
            torch.distributed.barrier()
        for s in range(warmup):
            tk = model.submit_train_step(seq[s], 0.2, grad_scale=1.0 / per)
            self.finish_step(self.start_allreduce(tk.gbuf), tk.gbuf)
            tk.result()
        torch.cuda.synchronize()
        if self.world > 1:
            torch.distributed.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t_p0 = time.perf_counter()
        packed = StepPrefetcher(model.pack_train_step, seq[warmup:], depth=2)        # loader thread, inside the timed region
        ticket = model.submit_train_step(next(packed), 0.2, grad_scale=1.0 / per)
        if trace is not None:
            print("[trace] loader start + first submit: %.2f ms" % ((time.perf_counter() - t_p0) * 1e3), file=sys.stderr)
        h2d = d2h = 0
        inflight, loss = [], torch.zeros(1)
        for s in range(warmup, n_steps):
            t_a = time.perf_counter()
            pending = self.start_allreduce(ticket.gbuf)
            t_1 = time.perf_counter()
            nb = next(packed) if s + 1 < n_steps else None
            t_2 = time.perf_counter()
            prep = model.prepare_train_step(nb) if nb is not None else None
            t_3 = time.perf_counter()
            self.finish_step(pending, ticket.gbuf)
            t_4 = time.perf_counter()
            nxt = prep.finish(0.2, grad_scale=1.0 / per) if prep is not None else None
            t_b = time.perf_counter()
            inflight.append(ticket)
            if len(inflight) > self.read_late:                   # the step's D2H read, `read_late` steps behind the enqueue front
                done = inflight.pop(0)
                loss, tsum = done.result()
                h2d += done.h2d_bytes
                d2h += done.d2h_bytes
            t_c = time.perf_counter()
            assert torch.isfinite(loss).all()
            t_d = time.perf_counter()
            ticket = nxt                                         # the finished step goes out of scope (slots, staging, gradient buffer)
            if trace is not None:      # all-reduce enqueue | packed batch from the loader thread | prepare | wait + Adam | finish | result wait | check | release
                trace.append((t_1 - t_a, t_2 - t_1, t_3 - t_2, t_4 - t_3, t_b - t_4, t_c - t_b, t_d - t_c, time.perf_counter() - t_d))
        for done in inflight:                                    # drain: every step's result is read inside the timed region
            loss, tsum = done.result()
            assert torch.isfinite(loss).all()
            h2d += done.h2d_bytes
            d2h += done.d2h_bytes
        e1.record()
        torch.cuda.synchronize()
        if trace is not None:
            print("[trace] e2e region %.2f ms for %d steps (host wall %.2f ms)" % (e0.elapsed_time(e1), steps, (time.perf_counter() - t_p0) * 1e3),
                  file=sys.stderr)
        return e0.elapsed_time(e1), sum(self.queries[s % len(self.steps)] for s in range(warmup, n_steps)), h2d, d2h



    def device_loop(self, *a, **k):
        with quiet_gc(self.model):
            return self._device_loop(*a, **k)

    def graph_loop(self, *a, **k):
        with quiet_gc(self.model):
            return self._graph_loop(*a, **k)

    def e2e_loop(self, *a, **k):
        with quiet_gc(self.model):
            return self._e2e_loop(*a, **k)

def dense_expansion_traffic(kg, cr, heads):
    """Bytes the expansion kernels MOVE in dense mode for the given slot heads -- a model of the kernel's own behaviour,
    counted from the graph (not the algorithmic figure): per trie node it reads the rows' pair-table pointers and entries
    (the in-edges whose source is a tail of the parent relation, as parent rows), pulls a parent row (128 B) per entry,
    and writes a row (128 B) only when at least one entry was pulled.  Both are
    static statistics of the (parent relation, relation) pair."""
    N, R = kg.entity_size, kg.relation_size
    h = kg.host
    dst_ptr, row_start, edge_src, row_dst = h["dst_ptr"], h["row_start"], h["edge_src"], h["row_dst"]
    is_tail = np.zeros((R, N), dtype=bool)
    for rho in range(R):
        is_tail[rho, row_dst[dst_ptr[rho]:dst_ptr[rho + 1]]] = True
    pulled = np.zeros((R, R), dtype=np.int64)           # [parent relation][relation]
    rows_w = np.zeros((R, R), dtype=np.int64)
    for rho in range(R):
        r0, r1 = int(dst_ptr[rho]), int(dst_ptr[rho + 1])
        if r1 == r0:
            continue
        e0, e1 = int(row_start[r0]), int(row_start[r1])
        M = is_tail[:, edge_src[e0:e1]]                 # [R, E_rho]
        pulled[:, rho] = M.sum(1)
        rows_w[:, rho] = np.logical_or.reduceat(M, (row_start[r0:r1] - e0).astype(np.int64), axis=1).sum(1)
    E, D = kg.rel_edges, kg.rel_rows
    node_rel, node_depth, node_head = cr.node_rel_host, cr.node_depth, cr.node_head
    prel = np.where(cr.host["node_parent"] >= 0, node_rel[np.maximum(cr.host["node_parent"], 0)], 0)
    root = node_depth == 1
    per_node = np.where(
        root, 4 * E[node_rel] + 8 * D[node_rel] + 128 * D[node_rel],             # depth 1: in-edges compared with h, every row written
        12 * D[node_rel] + 8 * pulled[prel, node_rel]                             # pair_ptr + row_dst per row, entry + bitmap word per pair entry
        + 128 * pulled[prel, node_rel] + 128 * rows_w[prel, node_rel])
    nb = np.zeros(cr.num_nodes + 1, dtype=np.int64)
    np.cumsum(per_node, out=nb[1:])
    head_bytes = nb[cr.head_node_ptr[1:]] - nb[cr.head_node_ptr[:-1]]
    return float(head_bytes[heads].sum())


def dump_outputs(out_dir, model, loss, tsum, gbuf):
    """What the last timed step hands its caller, as float32 DIR/<name>.npy: the loss and target sum of each batch, the
    gradients it accumulated and the parameters after its optimizer step (1.2 MB on the fb15k237 shape)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss, "target_sum": tsum, "rule_weights_grad": gbuf.view(model.rule_weights),
              "bias_grad": gbuf.view(model.bias), "rule_weights": model.rule_weights, "bias": model.bias}
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def reduce_max_sum(ms, q, dev, world):
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    n = torch.tensor([q], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        torch.distributed.all_reduce(n)
    return float(t.item()), float(n.item())


def deal_steps(batches, cr, per, n_distinct, world, rank, offset=0):
    """Every global step takes world*per batches and deals them to the ranks largest-first in snake order of
    their grounding cost (rows of the head's trie), so that the per-step all-reduce does not wait for one rank."""
    from rnnlogic_b200.trainer import snake_deal
    out = []
    for s in range(n_distinct):
        glob = [batches[(offset + s * per * world + j) % len(batches)] for j in range(per * world)]
        out.append([glob[j] for j in snake_deal([int(cr.head_rows[int(b[0, 1])]) for b in glob], world, rank)])
    return out


def rotate_dir(N, R, D=1000, gamma=9.0, seed=237):
    """BASELINE config 4: RotatE-shaped random entity features (hidden_dim 1000 -> eemb [N,2000], remb [R/2,1000])."""
    d = tempfile.mkdtemp(prefix="rotate_")
    rng = np.random.default_rng(seed)
    rr = (gamma + 2.0) / D
    np.save(os.path.join(d, "entity_embedding.npy"), rng.uniform(-rr, rr, size=(N, 2 * D)).astype(np.float32))
    np.save(os.path.join(d, "relation_embedding.npy"), rng.uniform(-rr, rr, size=(R // 2, D)).astype(np.float32))
    with open(os.path.join(d, "config.json"), "w") as f:
        json.dump({"hidden_dim": D, "gamma": gamma, "nentity": N}, f)
    return d


def side_config(tag, kg, rules, batches, kw, per, steps, world, rank, dev, plus=True, trace=False):
    """End-to-end train throughput of one more configuration (same loop as the headline's e2e)."""
    from rnnlogic_b200.predictors import Predictor, PredictorPlus
    torch.manual_seed(0)
    model = PredictorPlus(kg, **kw) if plus else Predictor(kg, **kw)
    model.set_rules([[h] + list(b) for h, b in rules])
    if not plus:
        g = torch.Generator().manual_seed(0)
        with torch.no_grad():
            model.rule_weights.copy_(torch.randn(model.num_rules, generator=g) * 0.1)
    model = model.cuda(dev)
    if plus and not model.supports_pipeline:
        return side_config_autograd(model, batches, per, steps, dev)
    if per == 1:                                     # reference schedule: per-head CUDA graphs
        run = Runner(model, deal_steps(batches, model.compiled, 1, 64, world, rank), 1, world, dev)
        ms, q = run.graph_loop(8, steps)
        ms, q = reduce_max_sum(ms, q, dev, world)
        out = {"e2e_queries_per_sec": q / (ms / 1e3), "ms_per_step": ms / steps, "steps": steps, "batches_per_step_per_gpu": 1,
               "path": "two CUDA graph replays (grounding of step k+1 behind the scoring of step k) + one event wait + one optimizer step per step; graphs captured once per head relation"}
        if rank == 0:
            print("[bench] %s: %.0f q/s e2e, %.3f ms/step" % (tag, out["e2e_queries_per_sec"], out["ms_per_step"]), file=sys.stderr)
        del run, model
        torch.cuda.empty_cache()
        return out
    run = Runner(model, deal_steps(batches, model.compiled, per, 4, world, rank), per, world, dev)
    run.size_cells()
    ms, q, h2d, d2h = run.e2e_loop(3, steps)
    ms, q = reduce_max_sum(ms, q, dev, world)
    out = {"e2e_queries_per_sec": q / (ms / 1e3), "ms_per_step": ms / steps, "steps": steps, "batches_per_step_per_gpu": per,
           "queries_per_step_per_gpu": int(np.mean(run.queries)), "h2d_bytes_per_step": h2d // steps, "d2h_bytes_per_step": d2h // steps}
    gr = run.sk.gr
    out["chunks_per_numeric_warp"] = {str(d): (gr.chunks_per_warp(d) or 16) for d in sorted(gr.level_density)}   # launch-shape feedback
    if rank == 0:
        print("[bench] %s: %.0f q/s e2e, %.3f ms/step (chunks per k_numeric warp by depth: %s)"
              % (tag, out["e2e_queries_per_sec"], out["ms_per_step"], out["chunks_per_numeric_warp"]), file=sys.stderr)
    del run, model
    torch.cuda.empty_cache()
    return out


def side_config_autograd(model, batches, per, steps, dev):
    """Configurations whose tail is not on the cell path yet (PNA aggregator): fused_train_step + torch optimizer."""
    popt = torch.optim.Adam(model.parameters(), lr=0.005)
    cycle = [[batches[(c * per + j) % len(batches)] for j in range(per)] for c in range(4)]
    st = {"i": 0}

    def step():
        sb = cycle[st["i"] % 4]
        st["i"] += 1
        popt.zero_grad(set_to_none=True)
        model.fused_train_step(sb, 0.2, grad_scale=1.0 / per)
        popt.step()

    for _ in range(4):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    q = sum(len(b) for sb in cycle for b in sb) / 4.0 * steps
    return {"e2e_queries_per_sec": q / (ms / 1e3), "ms_per_step": ms / steps, "steps": steps, "batches_per_step_per_gpu": per,
            "path": "autograd tail (PNA aggregator), host-synchronous"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--trace-e2e", action="store_true", help="print the host-side time of every end-to-end step to stderr")
    ap.add_argument("--batches", type=int, default=256, help="reference batches (of <=32 queries) per step per GPU")
    ap.add_argument("--dense", action="store_true", help="expand every row of every trie node (dense SpMM; roofline mode)")
    ap.add_argument("--dense-tail", action="store_true", help="round-1 tail (dense [S][N][32] logit / gradient matrices) for A/B")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the side configurations (configs / extras)")
    ap.add_argument("--only", default="", help="comma-separated side configurations to run (default: all)")
    ap.add_argument("--typed", action="store_true", help="headline on the typed synthetic graph instead of the i.i.d. one")
    ap.add_argument("--shape", default="fb15k237", choices=["fb15k237", "wn18rr"],
                    help="synthetic workload shape (the headline metric is quoted on fb15k237)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed headline step computed to DIR/<name>.npy "
                    "(inputs are seeded: two builds compare output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference" and rank != 0:
        return                                   # the CPU arm runs on rank 0 only; other ranks exit 0 without work
    shape, N, R, train, valid, test, rules = build_workload(args.shape, typed=args.typed)
    batches = make_batches(train, R, seed=1)
    per = args.batches
    workload = (shape["name"] + "-shape %s synthetic KG (N=%d, R=%d, E=%d train triples incl. inverses), %d synthetic rules "
                "of the reference rule file's shape (L<=%d), Predictor(bias) train step, B=32 per batch, %d batches per optimizer step per GPU"
                % ("typed" if args.typed else "i.i.d.", N, R, train.shape[0], len(rules), shape["max_len"], per))

    if args.impl == "reference":
        res = cpu_reference_run(N, R, train, valid, test, rules, batches, args.steps, args.warmup, per, budget_s=120.0)
        line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": res["steps_done"], "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/f32",
                "data": "synthetic", "config": {"workload": workload},
                "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    from rnnlogic_b200 import KnowledgeGraph
    from rnnlogic_b200.predictors import Predictor
    from rnnlogic_b200 import comm
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        comm.init_process_group("nccl", init_method="env://")

    kg = KnowledgeGraph(entity_size=N, relation_size=R, train=train, valid=valid, test=test)
    model = Predictor(kg, entity_feature="bias")
    model.force_dense = bool(args.dense)
    model.set_rules([[h] + list(b) for h, b in rules])
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        model.rule_weights.copy_(torch.randn(model.num_rules, generator=g) * 0.1)
    model = model.cuda(dev)
    cr = model.compiled
    n_distinct = args.warmup + args.steps
    run = Runner(model, deal_steps(batches, cr, per, n_distinct, world, rank), per, world, dev)
    sk = run.sk
    if args.dense_tail:                          # A/B: the round-1 dense tail behind the same loop
        def dense_step(sk_, sl, smoothing, scale, gbuf, bits=32, expanded=False):
            loss, tsum, _, gw, gb = model.step_on_slots_dense(sk_, sl, smoothing, scale, bits, expanded)
            gbuf.view(model.rule_weights).copy_(gw)
            gbuf.view(model.bias).copy_(gb)
            return loss, tsum
        model.step_on_slots = dense_step
        run.dense_tail = True
    run.size_cells()

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    # ---------------- device-resident timing (`value`) ----------------
    elapsed_ms, q_timed, launches, level_events = run.device_loop(args.warmup, args.steps, level_events=True)
    if args.dump_outputs and rank == 0:          # before the end-to-end loop trains the model further
        dump_outputs(args.dump_outputs, model, *run.last_step)
    step_ms_local = elapsed_ms
    elapsed_ms, q_total = reduce_max_sum(elapsed_ms, q_timed, dev, world)
    value = q_total / (elapsed_ms / 1e3)
    slots = run.slots

    # roofline of the dominant kernel (frontier expansion = k_symbolic + k_numeric per depth):
    # algorithmic bytes of SURVEY 8d for the timed heads / CUDA-event time of the expansion launches
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))

    def roofline_of(events, heads, step_ms, mode, note):
        exp_ms = {}
        for depth, e0, e1 in events:
            exp_ms[depth] = exp_ms.get(depth, 0.0) + e0.elapsed_time(e1)
        alg = float(cr.head_ground_bytes[heads].sum())
        n = len(events)
        tot = sum(exp_ms.values())
        ach = alg / (tot / 1e3) / 1e9 if tot > 0 else 0.0
        return {"bound": "hbm", "kernel": "frontier expansion (k_symbolic + k_numeric, all depths)", "mode": mode,
                "achieved": ach, "peak": peak, "peak_source": "measured" if "hbm_gbs" in peaks else "fallback",
                "unit": "GB/s", "frac": ach / peak, "traffic": None,
                "algorithmic_bytes_per_launch": alg / max(1, n), "avg_launch_ms": tot / max(1, n), "launches": n,
                "ms_by_depth": {str(k): v for k, v in sorted(exp_ms.items())}, "share_of_step": tot / step_ms,
                "note": note}

    n_steps = args.warmup + args.steps
    heads_timed = np.concatenate([slots[s].heads for s in range(args.warmup, n_steps)])
    roofline_product = roofline_of(
        level_events, heads_timed, step_ms_local, "dense SpMM" if model.force_dense else "sparse-aware (product path)",
        "rows that are provably all-zero are neither written nor read (exact); a fraction above 1 is sparsity "
        "exploitation, not bandwidth" if not model.force_dense else "every algorithmic byte is moved")
    roofline = roofline_product
    if not model.force_dense:
        # the same kernel as a plain dense SpMM on the same workload (every row of every trie node is
        # written and read, zeros included): the figure that says how close the kernel is to HBM
        sk.gr.force_dense = True
        nd = min(args.steps, 5)
        torch.cuda.synchronize()
        for s in range(3):
            sk.gr._run(slots[s], 32)
        torch.cuda.synchronize()
        sk.gr.level_events = []
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for s in range(args.warmup, args.warmup + nd):
            sk.gr._run(slots[s], 32)
        d1.record()
        torch.cuda.synchronize()
        dense_events, sk.gr.level_events = sk.gr.level_events, None
        sk.gr.force_dense = False
        heads_d = np.concatenate([slots[s].heads for s in range(args.warmup, args.warmup + nd)])
        roofline = roofline_of(dense_events, heads_d, d0.elapsed_time(d1), "dense expansion (force_dense), same kernel + workload",
                               "every row of every trie node is expanded (all in-edges examined); rows that are zero for "
                               "EVERY query and L2 hits keep DRAM traffic below the algorithmic bytes; the expansion alone, "
                               "timed in a second region right after the product loop (%d steps)" % nd)
        if rank == 0:
            # what the kernel itself moves in this mode (a parent row is pulled / a row written only where an in-edge starts at a
            # tail of the parent relation): the bandwidth figure; `frac` above credits the algorithmic bytes of SURVEY 8d
            moved = dense_expansion_traffic(kg, cr, heads_d)
            tot_ms = sum(float(v) for v in roofline["ms_by_depth"].values())
            roofline["moved_bytes_per_launch"] = moved / max(1, roofline["launches"])
            roofline["moved_bytes_source"] = "counted from the graph for this kernel's access pattern (bench.py: dense_expansion_traffic), not ncu"
            roofline["dram_frac"] = moved / (tot_ms / 1e3) / 1e9 / peak if tot_ms > 0 else None
            # measured DRAM bytes per launch of the same kernels in the same mode: one `ncu --set full` capture (profiles/),
            # valid for the default step size only -- a profiler cannot run inside a timed region
            tj = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_traffic.json")
            if os.path.exists(tj) and args.shape == "fb15k237" and not args.typed:
                with open(tj) as f:
                    tr = json.load(f)
                if int(tr.get("batches_per_step", -1)) == per:
                    roofline["traffic"] = float(tr["dram_bytes_per_launch"])
                    roofline["traffic_source"] = tr["source"]

    # ---------------- end-to-end through the public fused API (host arrays in, losses out) --------
    trace = [] if args.trace_e2e else None
    e2e_ms, q_e2e, h2d, d2h = run.e2e_loop(args.warmup, args.steps, trace)
    e2e_ms, q_e2e = reduce_max_sum(e2e_ms, q_e2e, dev, world)
    e2e_value = q_e2e / (e2e_ms / 1e3)
    if rank == 0:
        print("[bench] headline: value %.0f q/s (%.3f ms/step), e2e %.0f q/s, dense-mode roofline frac %.3f, expansion share %.2f"
              % (value, elapsed_ms / args.steps, e2e_value, roofline["frac"], roofline_product["share_of_step"]), file=sys.stderr)
    if args.trace_e2e and rank == 0:
        tr = np.asarray(trace) * 1e3
        print("e2e host ms per step [all-reduce enqueue | loader wait | prepare | nccl wait + Adam | finish | result wait | check | release]: median "
              + " ".join("%.3f" % v for v in np.median(tr, 0)) + " | mean " + " ".join("%.3f" % v for v in tr.mean(0))
              + " | max " + " ".join("%.3f" % v for v in tr.max(0)), file=sys.stderr)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32/f32", "data": "synthetic",
            "config": {"workload": workload, "queries_per_step_per_gpu": int(np.mean(run.queries)),
                       "l2_policy": "per-step working set (frontier arena %.1f GB) is larger than the 126 MB L2"
                                    % (float(cr.head_rows[heads_timed].sum()) * 128 / args.steps / 1e9),
                       "parallelism": "dp%d (queries sharded, KG replicated)" % world,
                       "dense_expansion": bool(model.force_dense), "tail": "dense Z/G matrices" if args.dense_tail else "candidate cells"},
            "roofline": roofline, "roofline_product": roofline_product,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d // args.steps,
                    "d2h_bytes_per_step": d2h // args.steps},
            "gpu_launches": int(launches)}

    # ---------------- the other configurations BASELINE.json names, same end-to-end loop ----------------
    if not args.no_extras:
        only = set(x for x in args.only.split(",") if x)
        want = lambda t: not only or t in only
        cfgs = {}
        side_steps = max(20, min(args.steps, 30))
        fb_plus = dict(type="lstm", num_layers=3, hidden_dim=16, entity_feature="bias", aggregator="sum")
        if want("reference_schedule_b1"):        # the reference's own schedule: ONE 32-query batch per optimizer step
            cfgs["reference_schedule_b1"] = side_config("b1", kg, rules, batches, dict(entity_feature="bias"), 1, 200, world, rank, dev, plus=False)
            cfgs["reference_schedule_b1"]["model"] = "Predictor(bias), 1 batch of <=32 queries per optimizer step (src/trainer.py:68-95)"
        if want("eval_filtered_rank"):
            tb = make_batches(test, R, seed=2)
            pe = min(per, 64)
            st = {"i": 0}

            def eval_step():
                sb = [tb[(st["i"] * pe + j) % len(tb)] for j in range(pe)]
                st["i"] += 1
                model.fused_rank(sb, "test")
                st["q"] = sum(len(b) for b in sb)

            for _ in range(3):
                eval_step()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(10):
                eval_step()
            a1.record()
            torch.cuda.synchronize()
            cfgs["eval_filtered_rank"] = {"e2e_queries_per_sec": st["q"] * 10 / (a0.elapsed_time(a1) / 1e3), "batches_per_call": pe,
                                          "model": "Predictor(bias): ground -> cells -> filtered rank (L,H)"}
        if want("fb15k237_plus_lstm_sum_bias"):  # config/FB15k-237_predictorplus.yaml
            cfgs["fb15k237_plus_lstm_sum_bias"] = side_config("plus", kg, rules, batches, fb_plus, per, side_steps, world, rank, dev)
            cfgs["fb15k237_plus_lstm_sum_bias"]["model"] = "PredictorPlus(lstm x3, sum, bias, H=16): the reference's shipped FB15k-237 config"
        if want("fb15k237_plus_lstm_sum_rotate1000"):   # BASELINE config 4
            kw = dict(fb_plus, entity_feature="RotatE", embedding_path=rotate_dir(N, R))
            p4 = min(per, 64)
            cfgs["fb15k237_plus_lstm_sum_rotate1000"] = side_config("rot", kg, rules, batches, kw, p4, side_steps, world, rank, dev)
            c4 = cfgs["fb15k237_plus_lstm_sum_rotate1000"]
            c4["model"] = "PredictorPlus(lstm, sum) + RotatE-shaped random entity feature D=1000 (BASELINE config 4)"
            flop = 13.0 * 32 * N * 1000 * 2.5                    # forward 13 B N D + backward ~1.5x, per 32-query batch
            c4["fp32_fraction"] = {"flop_per_batch": flop, "achieved_tflops": flop * p4 / (c4["ms_per_step"] / 1e3) / 1e12,
                                   "peak_tflops": 148 * 128 * 2 * 1.965e-3, "note": "RotatE epilogue is FP32/MUFU work: "
                                   "13*B*N*D flop forward (SURVEY 8d), ~1.5x that backward; peak = 148 SMs x 128 FMA lanes x 2 x 1.965 GHz"}
            c4["fp32_fraction"]["frac"] = c4["fp32_fraction"]["achieved_tflops"] / c4["fp32_fraction"]["peak_tflops"]
        del model, run
        torch.cuda.empty_cache()
        if want("fb15k237_typed_predictor_bias"):        # same sizes, rule bodies that compose
            _, tN, tR, ttrain, tvalid, ttest, trules = build_workload("fb15k237", typed=True)
            tkg = KnowledgeGraph(entity_size=tN, relation_size=tR, train=ttrain, valid=tvalid, test=ttest)
            tb_ = make_batches(ttrain, tR, seed=1)
            pt = min(per, 64)
            cfgs["fb15k237_typed_predictor_bias"] = side_config("typed", tkg, trules, tb_, dict(entity_feature="bias"), pt, side_steps, world, rank, dev, plus=False)
            cfgs["fb15k237_typed_predictor_bias"]["model"] = ("Predictor(bias) on a TYPED graph of the same sizes (12 entity types, every relation "
                                                             "has a domain/range, rule bodies are type-compatible chains): frontiers stay alive")
            if want("fb15k237_typed_plus_lstm_sum_bias"):
                cfgs["fb15k237_typed_plus_lstm_sum_bias"] = side_config("typedp", tkg, trules, tb_, fb_plus, pt, side_steps, world, rank, dev)
                cfgs["fb15k237_typed_plus_lstm_sum_bias"]["model"] = "PredictorPlus(lstm, sum, bias) on the typed graph"
            del tkg
        if want("wn18rr_plus_emb_pna_bias"):             # BASELINE config 3: config/wn18rr_predictorplus.yaml
            _, wN, wR, wtrain, wvalid, wtest, wrules = build_workload("wn18rr")
            wkg = KnowledgeGraph(entity_size=wN, relation_size=wR, train=wtrain, valid=wvalid, test=wtest)
            wb = make_batches(wtrain, wR, seed=1)
            pw = min(per, 64)
            cfgs["wn18rr_plus_emb_pna_bias"] = side_config("wn", wkg, wrules, wb, dict(type="emb", hidden_dim=16, entity_feature="bias", aggregator="pna"),
                                                           pw, side_steps, world, rank, dev)
            cfgs["wn18rr_plus_emb_pna_bias"]["model"] = "PredictorPlus(emb, pna, bias) on the WN18RR shape (BASELINE config 3)"
            if want("wn18rr_predictor_bias"):
                cfgs["wn18rr_predictor_bias"] = side_config("wnp", wkg, wrules, wb, dict(entity_feature="bias"), pw, side_steps, world, rank, dev, plus=False)
                cfgs["wn18rr_predictor_bias"]["model"] = "Predictor(bias) on the WN18RR shape (L<=5)"
            del wkg
        if want("scaled_1m_predictor_bias"):             # BASELINE config 5: 1M entities, 1k relations, 20M edges, 10k length-3 rules
            from rnnlogic_b200 import synth
            t_build = time.time()
            sN, sR, strain, svalid, stest = synth.scaled_kg()
            srules = synth.scaled_rules()
            skg = KnowledgeGraph(entity_size=sN, relation_size=sR, train=strain, valid=svalid, test=stest)
            sb = make_batches(strain[:2_000_000], sR, seed=1)    # batches from the first 2M facts (same relation mix)
            t_build = time.time() - t_build
            for pb in (64, 8):                                   # 2048 and 256 queries per optimizer step
                tag = "scaled_1m_predictor_bias" + ("" if pb == 64 else "_b%d" % (pb * 32))
                cfgs[tag] = side_config("scaled%d" % (pb * 32), skg, srules, sb, dict(entity_feature="bias"), pb, 10, world, rank, dev, plus=False)
                cfgs[tag]["model"] = ("Predictor(bias) on the scaled synthetic KG of BASELINE config 5 (N=1e6, R=1e3, E=2e7, 1e4 random "
                                      "length-3 rules), %d queries per optimizer step per GPU" % (pb * 32))
            cfgs["scaled_1m_predictor_bias"]["host_build_s"] = round(t_build, 1)
            del skg
        line["configs"] = cfgs

    clk = clocks.stop() if rank == 0 else None      # sampled over all timed regions
    line["clocks"] = clk
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    if world == 1 and not args.no_cpu_baseline:
        res = cpu_reference_run(N, R, train, valid, test, rules, batches, 1000, 1, per, budget_s=15.0)
        line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
