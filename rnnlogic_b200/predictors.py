"""Reasoning predictors with the reference's Python interface (src/predictors.py:17-271), running
on the hand-written sm_100a kernels.

``Predictor`` / ``PredictorPlus`` keep ``set_rules(list | path)``, ``forward(all_h, all_r,
edges_to_remove) -> (score fp32[B,N], mask bool[B,N])``, ``compute_H`` and the reference's
``state_dict`` keys.  They are CUDA-only: a CPU tensor raises (no fallback)."""
from __future__ import annotations

import ctypes as C
import logging
import math
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .engine import Grounder
from .hotpath import ScoreKernels
from .rules import CompiledRules, parse_rules

LANES = _lib.LANES


class _RuleModel(nn.Module):
    """Shared plumbing: rule parsing/compilation and per-device kernel drivers."""

    force_dense = False      # True: expand every row of every trie node (plain dense SpMM)

    def _load_rules(self, input, who):
        rules = parse_rules(input)
        logging.info("%s: read %d rules from %s." % (who, len(rules), "list" if type(input) == list else "file"))
        self.rules = [(h, b) for h, b in rules]
        self.num_rules = len(self.rules)
        self.relation2rules = [[] for _ in range(self.num_relations)]
        for index, rule in enumerate(self.rules):
            self.relation2rules[rule[0]].append([index, rule])
        self.compiled = CompiledRules(self.graph, self.rules)
        self._drivers = {}
        self.__dict__.pop("_graph_steps", None)        # captured per-head steps and rule-id tables belong to the old rule set
        self.__dict__.pop("_head_rule_ids", None)

    def _driver(self, device) -> ScoreKernels:
        if device.type != "cuda":
            raise _lib.RlError("rnnlogic_b200 predictors are CUDA-only (sm_100a); got a %s batch. There is no CPU "
                               "fallback: move the model and the batch to a CUDA device." % device)
        # the C-ABI entry points launch on the CURRENT device's stream: a model that lives on another GPU makes that GPU
        # current (one process per GPU is the design; this keeps `model.cuda(1); model(h, r, etr)` correct)
        if device.index is not None and device.index != torch.cuda.current_device():
            torch.cuda.set_device(device)
        key = str(device)
        if key not in self._drivers:
            self._drivers[key] = ScoreKernels(Grounder(self.graph, self.compiled, device, self.force_dense))
        return self._drivers[key]

    def _ground(self, all_h, all_r, edges_to_remove, coo_only=False):
        query_r = all_r[0].item()
        assert (all_r != query_r).sum() == 0
        sk = self._driver(all_r.device)
        sl = sk.gr.make_slots([query_r], [all_h.size(0)], all_h, None, edges_to_remove, coo_only=coo_only)
        sk.gr.ground(sl)
        return query_r, sk, sl


class Predictor(_RuleModel):
    """Linear rule-weight predictor (src/predictors.py:17-119)."""

    def __init__(self, graph, entity_feature="bias"):
        super(Predictor, self).__init__()
        self.graph = graph
        self.num_entities = graph.entity_size
        self.num_relations = graph.relation_size
        self.entity_feature = entity_feature
        if entity_feature == "bias":
            self.bias = nn.parameter.Parameter(torch.zeros(self.num_entities))

    def set_rules(self, input):
        self._load_rules(input, "Predictor")
        self.rule_weights = nn.parameter.Parameter(torch.zeros(self.num_rules, device=self._param_device()))

    def _param_device(self):
        return self.bias.device if self.entity_feature == "bias" else torch.device("cpu")

    def forward(self, all_h, all_r, edges_to_remove):
        query_r, sk, sl = self._ground(all_h, all_r, edges_to_remove, coo_only=True)
        use_bias = self.entity_feature == "bias"
        score, nz, n_cells = cellpath.predictor_api_scores(self, sk, sl)
        if n_cells == 0:                                                # predictors.py:67-71
            if use_bias:
                return score, torch.ones_like(nz)
            return torch.full_like(score, float("inf")), torch.zeros_like(nz)
        if use_bias:
            return score, torch.ones_like(nz)
        return score, nz

    @torch.no_grad()
    def compute_H(self, all_h, all_r, all_t, edges_to_remove):
        """E-step rule scores (src/predictors.py:82-119): per rule H = score[b,t] - mean over the
        batch's candidates of score[b,.], softmax over the head's rules, summed over the queries.
        The per-rule statistics come from one kernel (rl_rule_stats); no [R_q,B,N] tensor exists."""
        query_r = all_r[0].item()
        assert (all_r != query_r).sum() == 0
        device = all_r.device
        ids = self.compiled.head_rules[query_r]
        if len(ids) == 0:
            return None, None
        sk = self._driver(device)
        sl = sk.gr.make_slots([query_r], [all_h.size(0)], all_h, all_t.to(device), edges_to_remove, coo_only=True)
        sk.gr.ground(sl)
        sk.gr.build_cells(sl, 0, cap=1)               # for the candidate words sl.nzmask; the cell numbering is not read
        nzmask = sl.nzmask
        cr = self.compiled
        n_terms = max(1, int(cr.head_terms[query_r]))
        stats = torch.zeros(2, sl.S, n_terms, LANES, dtype=torch.float64, device=device)
        L = _lib.lib()
        _lib.check(L.rl_rule_stats(sk.dg.ref(), sk.dr.ref(), sl.ref(), sl.fref(), n_terms, stats[0].data_ptr(),
                                   stats[1].data_ptr(), _stream()), "rl_rule_stats")
        B = all_h.size(0)
        lanes = torch.arange(LANES, device=device, dtype=torch.int32)
        per_lane = ((nzmask.unsqueeze(-1) >> lanes) & 1).sum(1)                    # [S,32] candidates per query
        valid = torch.from_numpy(np.concatenate([s_ * LANES + np.arange(n) for s_, n in enumerate(sl.nq)])).to(device)
        neg_n = torch.clamp(per_lane.reshape(-1)[valid], min=1).to(torch.float32)    # [B]
        # [S,T,32] -> [B,T] in query order, then pick the head's rules in rule-file order
        to_q = lambda x: x.permute(0, 2, 1).reshape(sl.S * LANES, n_terms)[valid]
        sum_q, pos_q = to_q(stats[0]), to_q(stats[1])
        term_local = torch.from_numpy(np.where(cr.rule_nterm[ids] >= 0, cr.rule_nterm[ids] - cr.head_nterm0[query_r], -1)).to(device)
        has_body = term_local >= 0                                                   # empty-body rules: count = one_hot(h)
        tl = term_local.clamp(min=0)
        sum_c = torch.where(has_body.unsqueeze(0), sum_q[:, tl], torch.ones(B, len(ids), dtype=torch.float64, device=device))
        at_h = (all_h == all_t.to(device)).to(torch.float64).unsqueeze(1)
        pos_c = torch.where(has_body.unsqueeze(0), pos_q[:, tl], at_h.expand(B, len(ids)))
        w = self.rule_weights[torch.tensor(ids, device=device)].unsqueeze(0)
        pos_score = pos_c.float() * w
        neg_score = sum_c.float() * w / neg_n.unsqueeze(1)
        H = torch.softmax(pos_score - neg_score, dim=-1).sum(0)
        return H, torch.tensor(ids, dtype=torch.long, device=device)


# ------------------------------------------------------------------------------------------------
# fused paths used by rnnlogic_b200.trainer (no dense [B,N] target / flag tensors, no autograd)
# ------------------------------------------------------------------------------------------------
def _group_ptr(sl, device):
    """DEVICE int32[n_groups+1] slot ranges of the reference batches, or None when every batch fits
    one slot (then slot == group).  The table travels with the slot descriptors (engine.Slots)."""
    return sl.group_ptr_dev, len(sl.group_sizes)


_POP8 = torch.tensor([bin(i).count("1") for i in range(256)], dtype=torch.float32)


def _group_mask_sum(sl, nzmask, ng):
    """mask.sum() of each reference batch (trainer.py:87,96) from the per-entity lane bitmasks."""
    per_slot = _POP8.to(nzmask.device)[nzmask.view(torch.uint8).long()].view(sl.S, -1).sum(1)
    if ng == sl.S:
        return per_slot
    gid = torch.from_numpy(np.repeat(np.arange(ng), [(n + LANES - 1) // LANES for n in sl.group_sizes])).to(nzmask.device)
    return torch.zeros(ng, dtype=torch.float32, device=nzmask.device).index_add_(0, gid, per_slot)


def _predictor_step_on_slots_dense(self, sk, sl, smoothing, grad_scale=1.0, bits=32, expanded=False):
    """Round-1 tail kept for A/B measurements (bench.py --dense-tail): dense entity-major Z / G matrices
    [S][N][32] (rl_predictor_scores + rl_predictor_ce_backward).  Same results as the cell path."""
    device = sk.device
    use_bias = self.entity_feature == "bias"
    gptr, ng = _group_ptr(sl, device)
    if not expanded:
        sk.gr._run(sl, bits)
    gw = torch.zeros_like(self.rule_weights)
    gb = torch.zeros_like(self.bias) if use_bias else None
    scale = sk.slot_scale(sl.S, grad_scale)
    loss, tsum, nzmask = sk.predictor_train_tail(sl, self.rule_weights.detach(), self.bias.detach() if use_bias else None,
                                                 smoothing, gptr, ng, scale, gw, gb)
    msum = None if use_bias else _group_mask_sum(sl, nzmask, ng)
    return loss, tsum, msum, gw, gb


# ---- fused steps on candidate cells (cellpath.py): shared by Predictor and PredictorPlus -------------------
from . import cellpath  # noqa: E402


class RlStepOverflow(_lib.RlError):
    """An enqueued step must be redone: a path count did not fit 32 bits (redo with 64-bit rows) or the step had
    more candidate cells than its arrays hold (redo with larger arrays).  ``model.fused_train_step`` does both."""


def _fused_params(self):
    """Parameters the fused step writes gradients for, in a fixed order (= layout of the flat gradient buffer)."""
    return [p for p in self.parameters() if p.requires_grad]


def _step_on_slots(self, sk, sl, smoothing, grad_scale, gbuf, bits=32, expanded=False):
    """Enqueue one fused train step for prepared slots (no host sync); gradients accumulate into ``gbuf``.
    -> (loss[ng], tsum[ng]) device tensors."""
    if isinstance(self, Predictor):
        gb = gbuf.view(self.bias) if self.entity_feature == "bias" else None
        return cellpath.predictor_step(self, sk, sl, smoothing, grad_scale, gbuf.view(self.rule_weights), gb,
                                       expanded=expanded, bits=bits)
    return cellpath.plus_step(self, sk, sl, smoothing, grad_scale, gbuf, expanded=expanded, bits=bits)


def _dense_feature_params(self):
    if self.entity_feature == "bias":
        return [self.bias]
    if self.entity_feature == "RotatE":
        return [self.RotatE.eemb, self.RotatE.remb]
    return []


def _used_params(self, total_cells):
    """ids of the parameters that take part in a step (the others keep grad None, as under DDP's
    find_unused_parameters=True, trainer.py:60): without any candidate only the entity feature has a gradient
    (predictors.py:67-71, 230-237)."""
    if total_cells > 0:
        if isinstance(self, PredictorPlus):
            skip = [self.vocab_emb.weight] if self.type == "emb" else []
            return {id(p) for p in _fused_params(self) if all(p is not q for q in skip)}
        return {id(p) for p in _fused_params(self)}
    return {id(p) for p in _dense_feature_params(self)}


class _StepTicket:
    """Handle of an enqueued fused train step: everything is on the stream, nothing was synchronised.
    ``result()`` does the step's one device->host read (losses, target sums, cells per slot, flags)."""

    def __init__(self, model, sk, sl, batches, smoothing, grad_scale, loss, tsum, gbuf):
        self.model, self.sk, self.sl, self.batches = model, sk, sl, batches
        self.smoothing, self.grad_scale, self.gbuf = smoothing, grad_scale, gbuf
        self.ng = len(sl.group_sizes)
        pack = torch.cat([loss, tsum, sl.slot_ncell.float(), sl.flags.float()])
        self.pinned = torch.empty(pack.numel(), dtype=torch.float32, pin_memory=True)
        self.pinned.copy_(pack, non_blocking=True)
        self.event = torch.cuda.Event()
        self.event.record()
        self.h2d_bytes = sl.h2d_bytes
        self.d2h_bytes = int(pack.numel() * 4)
        self._done = None

    # gradients of the step (device), for loops that drive the optimizer themselves
    @property
    def gw(self):
        return self.gbuf.view(self.model.rule_weights)

    @property
    def gb(self):
        return self.gbuf.view(self.model.bias)

    def result(self):
        """(loss[n_batches], target_sum[n_batches]) host tensors.  Raises RlStepOverflow when the step has to be redone."""
        if self._done is not None:
            return self._done
        self.event.synchronize()
        host, ng, S = self.pinned, self.ng, self.sl.S
        flags = host[2 * ng + S:]                           # cell counters[8] | count overflow | non-zero rows per depth[8]
        self.total_cells = int(flags[0].item())
        self.sk.gr.note_cell_count(self.total_cells)
        self.sk.gr.note_level_rows(self.sl, flags[9:17].tolist())
        self.count_overflow = flags[8].item() != 0
        if self.count_overflow:
            raise RlStepOverflow("a path count overflowed 32 bits inside an enqueued step; redo it with "
                                 "model.fused_train_step (exact 64-bit rows)")
        if flags[1].item() != 0:
            raise RlStepOverflow("the step has %d candidate cells, more than its arrays hold; redo it with "
                                 "model.fused_train_step (the arrays grow)" % self.total_cells)
        ncell = host[2 * ng:2 * ng + S].numpy()
        gslots = [(n + LANES - 1) // LANES for n in self.sl.group_sizes]
        self.mask_sum = np.add.reduceat(ncell, np.concatenate([[0], np.cumsum(gslots)[:-1]])).tolist() if S else []
        dense_feature = self.model.entity_feature in ("bias", "RotatE")
        self.model.last_mask_sum = None if dense_feature else self.mask_sum
        self.used = _used_params(self.model, self.total_cells)
        self._done = (host[:ng], host[ng:2 * ng])
        return self._done


class _PreparedStep:
    """The parameter-independent half of a fused train step, already enqueued: host pack -> one H2D ->
    slot preparation -> frontier expansion.  ``finish()`` enqueues the parameter-dependent half."""

    def __init__(self, model, sk, sl, batches, bits):
        self.model, self.sk, self.sl, self.batches, self.bits = model, sk, sl, batches, bits

    def finish(self, smoothing, grad_scale=1.0):
        """cells -> scores -> CE -> backward -> async D2H of the losses; returns the step's ticket."""
        model, sk, sl = self.model, self.sk, self.sl
        gbuf = cellpath.GradBuffer(_fused_params(model))
        loss, tsum = _step_on_slots(model, sk, sl, smoothing, grad_scale, gbuf, self.bits, expanded=True)
        return _StepTicket(model, sk, sl, self.batches, smoothing, grad_scale, loss, tsum, gbuf)


def _model_device(self):
    return next(self.parameters()).device


def _pack_train(self, batches):
    """The CUDA-free part of a fused train step (queries and slot tables packed into pinned memory for one
    copy).  Thread-safe once the model sits on its device: a loader thread can pack steps ahead
    (data.StepPrefetcher) and hand the result to prepare_train_step / submit_train_step."""
    return self._driver(_model_device(self)).gr.pack_host(batches, with_etr=True)


def _prepare_train(self, batches):
    """Enqueue everything of a fused train step that does not depend on the parameters (grounding) and
    return a handle; ``handle.finish(smoothing, grad_scale)`` enqueues the rest.  A data-parallel loop calls
    this for step k+1 while the gradient all-reduce of step k is in flight.  ``batches``: a list of
    single-relation batches or a step packed ahead by pack_train_step."""
    sk = self._driver(_model_device(self))
    sl = sk.gr.make_slots_host(batches, with_etr=True, coo_only=True)
    bits = sk.gr.force_bits or 32
    sk.gr._run(sl, bits)
    return _PreparedStep(self, sk, sl, batches, bits)


def _submit_train(self, batches, smoothing, grad_scale=1.0):
    """Enqueue one fused train step (host pack -> H2D -> kernels -> async D2H) and return a ticket; the
    gradients are in ticket.gbuf (device).  Lets the host prepare step k+1 while step k runs."""
    return _prepare_train(self, batches).finish(smoothing, grad_scale)


def _fused_train(self, batches, smoothing, grad_scale=1.0):
    """One fused step over a list of single-relation train batches (trainer.py:68-93 for each):
    ground -> cells -> scores -> log(softmax+1e-8) CE -> backward.  Gradients of ``grad_scale * sum of
    the batch losses`` are ACCUMULATED into .grad (parameters that did not take part keep None).  Returns
    (loss[n_batches], target_sum[n_batches]) as host float tensors -- one device->host read per step.
    A 32-bit count overflow redoes the step with 64-bit rows, a cell-array overflow with larger arrays."""
    sk = self._driver(_model_device(self))
    host = batches if not isinstance(batches, list) else sk.gr.pack_host(batches, with_etr=True)
    bits = sk.gr.force_bits or 32
    for _attempt in range(10):
        sl = sk.gr.make_slots_host(host, with_etr=True, coo_only=True)
        sk.gr._run(sl, bits)
        ticket = _PreparedStep(self, sk, sl, batches, bits).finish(smoothing, grad_scale)
        try:
            loss, tsum = ticket.result()
            break
        except RlStepOverflow:
            if ticket.count_overflow:                      # exact 64-bit rows (they wrap like the reference's int64)
                bits = 64
    else:
        raise _lib.RlError("fused_train_step: the cell arrays kept overflowing")
    for p in _fused_params(self):
        if id(p) in ticket.used:
            g = ticket.gbuf.view(p)
            p.grad = g if p.grad is None else p.grad.add_(g)
    self.last_h2d_bytes = sl.h2d_bytes
    self.last_d2h_bytes = ticket.d2h_bytes
    self.last_ticket = ticket
    return loss, tsum


@torch.no_grad()
def _fused_rank(self, batches, split):
    """(L,H) int64[Q,2] of a list of single-relation eval batches (trainer.py:173,189-201)."""
    sk = self._driver(_model_device(self))
    sl = sk.gr.make_slots_host(batches, with_etr=False, coo_only=True)
    if isinstance(self, Predictor):
        LH = cellpath.predictor_rank(self, sk, sl, split)
    else:
        LH = cellpath.plus_rank(self, sk, sl, split)
    return _valid_lanes(sl, LH)


def _valid_lanes(sl, LH):
    idx = np.concatenate([s * LANES + np.arange(n) for s, n in enumerate(sl.nq)])
    return LH[torch.from_numpy(idx).to(LH.device)]


def _install_fused(cls):
    cls.fused_train_step = _fused_train
    cls.submit_train_step = _submit_train
    cls.prepare_train_step = _prepare_train
    cls.pack_train_step = _pack_train
    cls.step_on_slots = _step_on_slots
    cls.fused_rank = _fused_rank
    cls.fused_params = _fused_params


_install_fused(Predictor)
Predictor.step_on_slots_dense = _predictor_step_on_slots_dense


# ================================================================================================
# PredictorPlus (src/predictors.py:121-271)
# ================================================================================================
from .layers import MLP, FuncToNode, FuncToNodeSum  # noqa: E402
from .engine import _stream  # noqa: E402


class _PlusCtx:
    """Everything the PredictorPlus kernels of one call share."""

    def __init__(self, sk, sl, H, pna):
        self.sk, self.sl, self.H, self.pna = sk, sl, H, pna
        dev = sk.device
        N, S = sk.N, sl.S
        self.nzmask = torch.empty(S, N, dtype=torch.int32, device=dev)
        cand_cnt = torch.empty(S * N, dtype=torch.int32, device=dev)
        _lib.check(_lib.lib().rl_plus_mask(sk.dg.ref(), sk.dr.ref(), sl.ref(), sl.fref(), self.nzmask.data_ptr(),
                                           cand_cnt.data_ptr(), _stream()), "rl_plus_mask")
        csum = torch.cumsum(cand_cnt, 0, dtype=torch.int64)
        self.cand_off = (csum - cand_cnt).contiguous()
        self.C = int(csum[-1].item())                     # host sync, as torch.nonzero in predictors.py:239
        self.rule_local = None
        self.arg_min = self.arg_max = None


class _PlusAggregateFn(torch.autograd.Function):
    """emb[n,H] -> per-candidate statistics (kernel rl_plus_features) with the backward into emb
    (kernel rl_plus_backward).  sum: (F,) ; pna: (S1, S2, MN, MX)."""

    @staticmethod
    def forward(ctx, emb, pc):
        sk, sl, H, C = pc.sk, pc.sl, pc.H, pc.C
        dev = emb.device
        embc = emb.detach().contiguous().float()
        n_out = 4 if pc.pna else 1
        out = torch.empty(n_out, C, H, dtype=torch.float32, device=dev)
        pc.cand_query = torch.empty(C, dtype=torch.int64, device=dev)
        pc.degree = torch.empty(C, dtype=torch.float32, device=dev) if pc.pna else None
        if pc.pna:
            pc.arg_min = torch.empty(C, H, dtype=torch.int32, device=dev)
            pc.arg_max = torch.empty(C, H, dtype=torch.int32, device=dev)
        _lib.check(_lib.lib().rl_plus_features(
            sk.dg.ref(), sk.dr.ref(), sl.ref(), sl.fref(), pc.nzmask.data_ptr(), pc.cand_off.data_ptr(),
            sl.q_off_dev.data_ptr(), pc.rule_local.data_ptr(), embc.data_ptr(), H, int(pc.pna),
            out[0].data_ptr(), out[1].data_ptr() if pc.pna else None, out[2].data_ptr() if pc.pna else None,
            out[3].data_ptr() if pc.pna else None, pc.arg_min.data_ptr() if pc.pna else None,
            pc.arg_max.data_ptr() if pc.pna else None, pc.degree.data_ptr() if pc.pna else None,
            pc.cand_query.data_ptr(), _stream()), "rl_plus_features")
        ctx.pc = pc
        ctx.save_for_backward(embc)
        return tuple(out[i] for i in range(n_out))

    @staticmethod
    def backward(ctx, *grads):
        pc = ctx.pc
        (embc,) = ctx.saved_tensors
        sk, sl, H = pc.sk, pc.sl, pc.H
        dA = grads[0].contiguous().float()
        dB = grads[1].contiguous().float() if pc.pna else None
        gA = torch.zeros_like(embc)
        gB = torch.zeros_like(embc) if pc.pna else None
        max_terms = int(sk.cr.head_terms[sl.heads].max())
        _lib.check(_lib.lib().rl_plus_backward(
            sk.dg.ref(), sk.dr.ref(), sl.ref(), sl.fref(), pc.nzmask.data_ptr(), pc.cand_off.data_ptr(),
            pc.rule_local.data_ptr(), H, dA.data_ptr(), dB.data_ptr() if dB is not None else None, max_terms,
            gA.data_ptr(), gB.data_ptr() if gB is not None else None, _stream()), "rl_plus_backward")
        g = gA
        if pc.pna:
            g = g + 2.0 * embc * gB                       # d/d emb of sum count * emb^2
            cols = torch.arange(H, device=g.device).unsqueeze(0)
            flat = g.view(-1)
            for arg, dv in ((pc.arg_min, grads[2]), (pc.arg_max, grads[3])):   # min/max route to their arg rule
                flat.index_add_(0, (arg.long() * H + cols).view(-1), dv.contiguous().view(-1).float())
        return g, None


class _PlusScatterFn(torch.autograd.Function):
    """candidate scores (+ bias, + entity-feature logits) -> entity-major logits Z[S][N][32]."""

    @staticmethod
    def forward(ctx, zc, bias, extra, pc, fill_neg_inf):
        sk, sl = pc.sk, pc.sl
        Z = torch.empty(sl.S, sk.N, LANES, dtype=torch.float32, device=sk.device)
        zcc = zc.detach().contiguous().float() if zc is not None else torch.zeros(1, device=sk.device)
        bc = bias.detach().contiguous() if bias is not None else None       # held in locals until the call is enqueued
        ec = extra.detach().contiguous() if extra is not None else None
        _lib.check(_lib.lib().rl_plus_scatter(
            sk.dg.ref(), sl.ref(), pc.nzmask.data_ptr(), pc.cand_off.data_ptr(), zcc.data_ptr(),
            bc.data_ptr() if bc is not None else None,
            ec.data_ptr() if ec is not None else None, int(fill_neg_inf),
            Z.data_ptr(), _stream()), "rl_plus_scatter")
        ctx.pc = pc
        ctx.flags = (zc is not None, bias is not None, extra is not None)
        return Z

    @staticmethod
    def backward(ctx, G):
        pc = ctx.pc
        sk, sl = pc.sk, pc.sl
        has_z, has_b, has_x = ctx.flags
        G = G.contiguous()
        dz = db = None
        if has_z:
            dz = torch.zeros(max(1, pc.C), dtype=torch.float32, device=G.device)
            _lib.check(_lib.lib().rl_plus_gather(sk.dg.ref(), sl.ref(), pc.nzmask.data_ptr(), pc.cand_off.data_ptr(),
                                                 G.data_ptr(), dz.data_ptr(), _stream()), "rl_plus_gather")
            dz = dz[:pc.C]
        if has_b:
            # NaN-safe: cells filled with -inf never coexist with a bias (mask mode has none)
            db = G.sum(dim=(0, 2))
        return dz, db, (G if has_x else None), None, None


class _ToDenseFn(torch.autograd.Function):
    """entity-major Z[S][N][32] -> the reference's [B,N] layout (and back for the gradient)."""

    @staticmethod
    def forward(ctx, Z, nzmask, sk, sl):
        score, nz = sk.to_dense(sl, Z.contiguous(), nzmask)
        ctx.sk, ctx.sl = sk, sl
        ctx.mark_non_differentiable(nz)
        return score, nz

    @staticmethod
    def backward(ctx, gscore, _gnz):
        return ctx.sk.from_dense(ctx.sl, gscore.contiguous()), None, None, None


class _LstmEncodeFn(torch.autograd.Function):
    """torch.nn.LSTM(H, H, L, batch_first=True)(x)[0] gathered at the last non-pad step, on the hand-written
    kernels of rl_rnn.cu (the sequential part) + one GEMM per weight gradient."""

    @staticmethod
    def forward(ctx, x, lens, L, *weights):
        n, T, H = x.shape
        x = x.contiguous().float()
        weights = [w.detach().contiguous().float() for w in weights]
        dev = x.device
        acts = torch.zeros(n, L, T, 5, H, dtype=torch.float32, device=dev)
        ih = torch.zeros(L, n, T, 2 * H, dtype=torch.float32, device=dev)
        out = torch.empty(n, H, dtype=torch.float32, device=dev)
        ptrs = (C.c_void_p * (4 * L))(*[w.data_ptr() for w in weights])
        _lib.check(_lib.lib().rl_lstm_encode_forward(n, T, H, L, x.data_ptr(), lens.data_ptr(), ptrs, acts.data_ptr(),
                                                     ih.data_ptr(), out.data_ptr(), _stream()), "rl_lstm_encode_forward")
        ctx.save_for_backward(lens, acts, ih, *weights)
        ctx.shape = (n, T, H)
        ctx.L = L
        return out

    @staticmethod
    def backward(ctx, dout):
        lens, acts, ih, *weights = ctx.saved_tensors
        L = ctx.L
        n, T, H = ctx.shape
        dev = acts.device
        dG = torch.zeros(L, n, T, 4 * H, dtype=torch.float32, device=dev)
        dX = torch.zeros(n, T, H, dtype=torch.float32, device=dev)
        ptrs = (C.c_void_p * (4 * L))(*[w.data_ptr() for w in weights])
        _lib.check(_lib.lib().rl_lstm_encode_backward(n, T, H, L, lens.data_ptr(), ptrs, acts.data_ptr(),
                                                      dout.contiguous().float().data_ptr(), dG.data_ptr(), dX.data_ptr(),
                                                      _stream()), "rl_lstm_encode_backward")
        # plain reductions over (rule, step): [dW_ih | dW_hh] = dG^T ih and the bias sums, one kernel for all layers
        dW = torch.zeros(L, 4 * H, 2 * H, dtype=torch.float32, device=dev)
        db = torch.zeros(L, 4 * H, dtype=torch.float32, device=dev)
        _lib.check(_lib.lib().rl_lstm_encode_wgrad(n * T, H, L, dG.data_ptr(), ih.data_ptr(), dW.data_ptr(), db.data_ptr(),
                                                   _stream()), "rl_lstm_encode_wgrad")
        grads = []
        for l in range(L):
            grads += [dW[l, :, :H], dW[l, :, H:], db[l], db[l]]
        return (dX, None, None) + tuple(grads)


class PredictorPlus(_RuleModel):
    fused_rnn = True          # `lstm` rule encoder with hidden_dim 16 / 32: rl_rnn.cu instead of cuDNN

    def __init__(self, graph, type='emb', num_layers=3, hidden_dim=16, entity_feature='bias', aggregator='sum',
                 embedding_path=None):
        super(PredictorPlus, self).__init__()
        self.graph = graph
        self.type = type
        self.num_layers = num_layers
        self.hidden_dim = hidden_dim
        self.entity_feature = entity_feature
        self.aggregator = aggregator
        self.embedding_path = embedding_path
        self.num_entities = graph.entity_size
        self.num_relations = graph.relation_size
        self.padding_index = graph.relation_size
        self._scratch = {}
        self.vocab_emb = torch.nn.Embedding(self.num_relations + 1, self.hidden_dim, padding_idx=self.num_relations)
        own_lstm = self.type == 'lstm' and self.fused_rnn and self.hidden_dim in (16, 32) and 1 <= self.num_layers <= 4
        if self.type in ('lstm', 'gru', 'rnn') and not own_lstm:
            # Only the encoders that run on cuDNN touch this process-global switch (the shipped lstm configs run on
            # rl_rnn.cu and leave it alone): cuDNN RNNs default to TF32 matmuls, forward AND backward; the rule encoder
            # must stay in true fp32 for the 1e-5 parity bar, and the backward runs outside any context manager.
            torch.backends.cudnn.allow_tf32 = False
        if self.type == 'lstm':
            self.rnn = torch.nn.LSTM(self.hidden_dim, self.hidden_dim, self.num_layers, batch_first=True)
        elif self.type == 'gru':
            self.rnn = torch.nn.GRU(self.hidden_dim, self.hidden_dim, self.num_layers, batch_first=True)
        elif self.type == 'rnn':
            self.rnn = torch.nn.RNN(self.hidden_dim, self.hidden_dim, self.num_layers, batch_first=True)
        elif self.type == 'emb':
            self.rule_emb = None
        else:
            raise NotImplementedError
        if aggregator == 'sum':
            self.rule_to_entity = FuncToNodeSum(self.hidden_dim)
        elif aggregator == 'pna':
            self.rule_to_entity = FuncToNode(self.hidden_dim)
        else:
            raise NotImplementedError
        self.relation_emb = torch.nn.Embedding(self.num_relations, self.hidden_dim)
        self.score_model = MLP(self.hidden_dim * 2, [128, 1])
        if entity_feature == 'bias':
            self.bias = torch.nn.parameter.Parameter(torch.zeros(self.num_entities))
        elif entity_feature == 'RotatE':
            from .embedding import RotatE
            self.RotatE = RotatE(embedding_path)

    def set_rules(self, input):
        self._load_rules(input, "Predictor+")
        self.max_length = max([len(rule[1]) for rule in self.rules])
        feats = [[h] + list(b) + [self.padding_index] * (self.max_length - len(b)) for h, b in self.rules]
        self.rule_features = torch.tensor(feats, dtype=torch.long)
        if self.type == 'emb':
            dev = self.relation_emb.weight.device
            self.rule_emb = nn.parameter.Parameter(torch.zeros(self.num_rules, self.hidden_dim, device=dev))
            nn.init.kaiming_uniform_(self.rule_emb, a=math.sqrt(5), mode="fan_in")

    def _emb_scratch(self, device, grad=False):
        """[num_rules, H] fp32 scratch indexed by the global rule id (rule embeddings of a step / their gradient)."""
        key = ("g" if grad else "e") + str(device)
        t = self._scratch.get(key)
        if t is None or t.shape[0] != self.num_rules:
            t = self._scratch[key] = torch.zeros(self.num_rules, self.hidden_dim, dtype=torch.float32, device=device)
        return t

    def _d1sum_scratch(self, device):
        key = "d" + str(device)
        t = self._scratch.get(key)
        if t is None:
            n = int(_lib.lib().rl_tail_scratch_floats(self.num_relations))
            t = self._scratch[key] = torch.empty(n, dtype=torch.float32, device=device)
        return t

    def encode_rules(self, rule_features):
        """predictors.py:201-208: embed [head, body..., pad], run the RNN, take the last non-pad output."""
        rule_masks = rule_features != self.num_relations
        x = self.vocab_emb(rule_features)
        if (self.fused_rnn and self.type == 'lstm' and x.is_cuda and self.hidden_dim in (16, 32)
                and 1 <= self.num_layers <= 4 and x.shape[0] > 0):
            ws = [getattr(self.rnn, "%s_l%d" % (nm, l)) for l in range(self.num_layers)
                  for nm in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
            return _LstmEncodeFn.apply(x, rule_masks.sum(-1).to(torch.int32), self.num_layers, *ws)
        output, hidden = self.rnn(x)
        idx = (rule_masks.sum(-1) - 1).long()
        idx = idx.unsqueeze(-1).unsqueeze(-1).expand(-1, -1, self.hidden_dim)
        return torch.gather(output, 1, idx).squeeze(1)

    # ---- the shapes the cell kernels do not take (cellpath.plus_cells_supported): forward and fused steps ----
    def _logits(self, sk, sl):
        """Z[S][N][32] (autograd-connected to every parameter), nzmask[S][N]."""
        device = sk.device
        H = self.hidden_dim
        ef = self.entity_feature
        pc = _PlusCtx(sk, sl, H, self.aggregator == 'pna')
        zc = None
        if pc.C > 0:
            heads = sorted(set(int(h) for h in sl.heads))
            rule_ids = torch.tensor([i for q in heads for i in self.compiled.head_rules[q]], dtype=torch.long,
                                    device=device)
            pc.rule_local = torch.full((self.num_rules,), -1, dtype=torch.int32, device=device)
            pc.rule_local[rule_ids] = torch.arange(rule_ids.numel(), dtype=torch.int32, device=device)
            if self.type == 'emb':
                emb = self.rule_emb[rule_ids]
            else:
                if self.rule_features.device != device:
                    self.rule_features = self.rule_features.to(device)
                emb = self.encode_rules(self.rule_features[rule_ids])
            stats = _PlusAggregateFn.apply(emb, pc)
            qhead = torch.from_numpy(np.repeat(sl.heads, sl.nq)).to(device)
            cand_head = qhead[pc.cand_query]
            if self.aggregator == 'sum':
                out = self.rule_to_entity.post(stats[0])
            else:
                out = self.rule_to_entity.post(stats[0], stats[1], stats[2], stats[3], pc.degree, pc.cand_query,
                                               int(sl.q_off[-1]))
            rel = self.relation_emb(cand_head)
            zc = self.score_model(torch.cat([out, rel], dim=-1)).squeeze(-1)
        bias = self.bias if ef == 'bias' else None
        extra = self.RotatE.slot_scores(sk, sl) if ef == 'RotatE' else None
        Z = _PlusScatterFn.apply(zc, bias, extra, pc, ef not in ('bias', 'RotatE'))
        return Z, pc

    def forward(self, all_h, all_r, edges_to_remove):
        if cellpath.plus_cells_supported(self):
            query_r, sk, sl = self._ground(all_h, all_r, edges_to_remove, coo_only=True)
            score, nz, n_cells = cellpath.plus_api_scores(self, sk, sl)
        else:
            query_r, sk, sl = self._ground(all_h, all_r, edges_to_remove)
            Z, pc = self._logits(sk, sl)
            score, nz = _ToDenseFn.apply(Z, pc.nzmask, sk, sl)
            n_cells = pc.C
        dense_feature = self.entity_feature in ('bias', 'RotatE')
        if n_cells == 0 and not dense_feature:                           # predictors.py:236-237
            return torch.full_like(score, float("inf")), torch.zeros_like(nz)
        if dense_feature:
            return score, torch.ones_like(nz)
        return score, nz


def _plus_fused_train(self, batches, smoothing, grad_scale=1.0):
    """Fused train step for PredictorPlus: CUDA grounding / aggregation / CE, torch autograd only for
    the small dense tail (rule encoder, Linear/LayerNorm/MLP on the C candidate rows)."""
    device = self.relation_emb.weight.device
    sk = self._driver(device)
    use_mask = self.entity_feature not in ('bias', 'RotatE')
    sl = sk.gr.make_slots_host(batches, with_etr=True)    # frontier in the reusable workspace: the autograd
    gptr, ng = _group_ptr(sl, device)                     # backward below runs before this call returns
    sk.gr.ground(sl)
    Z, pc = self._logits(sk, sl)
    loss, tsum, G = sk.softmax_ce(sl, Z.detach(), pc.nzmask, smoothing, use_mask, gptr, ng, want_grad=True)
    if grad_scale != 1.0:
        G = G * grad_scale
    if Z.requires_grad:
        Z.backward(G)
    parts = [loss, tsum] + ([_group_mask_sum(sl, pc.nzmask, ng)] if use_mask else [])
    host = torch.cat(parts).cpu()
    self.last_h2d_bytes = sl.h2d_bytes
    self.last_d2h_bytes = int(host.numel() * 4) + 8
    self.last_mask_sum = host[2 * ng:3 * ng].tolist() if use_mask else None
    return host[:ng], host[ng:2 * ng]


@torch.no_grad()
def _plus_fused_rank(self, batches, split):
    device = self.relation_emb.weight.device
    sk = self._driver(device)
    use_mask = self.entity_feature not in ('bias', 'RotatE')
    sl = sk.gr.make_slots_host(batches, with_etr=False)
    sk.gr.ground(sl)
    Z, pc = self._logits(sk, sl)
    LH = sk.filtered_rank(sl, Z.contiguous(), pc.nzmask, "hr2oo" if split == "valid" else "hr2ooo", use_mask)
    return _valid_lanes(sl, LH)


_install_fused(PredictorPlus)


def _plus_train_dispatch(self, batches, smoothing, grad_scale=1.0):
    """Cell path (hand-written backward, no host sync) for the sum aggregator at hidden_dim 16; the PNA aggregator
    and other widths take the autograd path above."""
    if cellpath.plus_cells_supported(self):
        return _fused_train(self, batches, smoothing, grad_scale)
    return _plus_fused_train(self, batches, smoothing, grad_scale)


def _plus_rank_dispatch(self, batches, split):
    if cellpath.plus_cells_supported(self):
        return _fused_rank(self, batches, split)
    return _plus_fused_rank(self, batches, split)


PredictorPlus.fused_train_step = _plus_train_dispatch
PredictorPlus.fused_rank = _plus_rank_dispatch
Predictor.supports_pipeline = property(lambda self: True)
PredictorPlus.supports_pipeline = property(lambda self: cellpath.plus_cells_supported(self))
