"""Fused train / eval steps on candidate cells (csrc/rl_cells.cu, rl_tail_tc.cu): what TrainerPredictor and
bench.py run.  Nothing of size [B,N] is built; no host synchronisation happens inside a step -- the
candidate count stays on the device (the reference syncs on it four times per batch,
src/predictors.py:211,230,239, src/layers.py:65) and comes back with the losses in the step's one D2H read.

Reference semantics: Predictor.forward / PredictorPlus.forward (src/predictors.py:53-80, 210-271) +
the loss of TrainerPredictor.train (src/trainer.py:84-93) + the rank of evaluate (src/trainer.py:189-201)."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import numpy as np
import torch

from . import _lib
from .engine import _stream

LANES = _lib.LANES
_L = _lib.lib


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


class GradBuffer:
    """One flat fp32 gradient buffer with a view per parameter: kernels accumulate into the views, the
    data-parallel exchange all-reduces ``flat`` directly (no torch.cat per step)."""

    def __init__(self, params: List[torch.nn.Parameter]):
        self.params = list(params)
        sizes = [p.numel() for p in self.params]
        offs = np.concatenate([[0], np.cumsum([(n + 3) // 4 * 4 for n in sizes])])     # 16-byte aligned views
        dev = self.params[0].device
        self.flat = torch.zeros(int(offs[-1]), dtype=torch.float32, device=dev)
        self.views = [self.flat[int(o):int(o) + n].view_as(p) for o, n, p in zip(offs[:-1], sizes, self.params)]
        self.of = {id(p): v for p, v in zip(self.params, self.views)}

    def view(self, p):
        return self.of[id(p)]

    def assign(self, used=None):
        """p.grad = its view (parameters not in ``used`` keep grad None: DDP find_unused_parameters semantics)."""
        for p, v in zip(self.params, self.views):
            p.grad = v if (used is None or id(p) in used) else None


class CellKernels:
    """ctypes drivers of the cell kernels for one ScoreKernels (= one device)."""

    def __init__(self, sk):
        self.sk = sk
        self.gr, self.dg, self.dr = sk.gr, sk.dg, sk.dr
        self.N, self.device = sk.N, sk.device
        self.acc = torch.zeros(4, dtype=torch.float64, device=self.device)       # Mg, Sg, K

    def bias_stats(self, bias: torch.Tensor):
        _lib.check(_L().rl_bias_stats(self.N, bias.data_ptr(), self.acc.data_ptr(), _stream()), "rl_bias_stats")

    def predictor_scores(self, sl, w, zc):
        _lib.check(_L().rl_predictor_item_scores(self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), C.byref(sl.cells),
                                                w.data_ptr(), zc.data_ptr(), _stream()), "rl_predictor_item_scores")

    def softmax_ce(self, sl, bias, zc, smoothing, group_ptr, n_groups, grad_scale, Gc, grad_bias):
        """-> (group_loss, group_tsum) device tensors; Gc / grad_bias filled when Gc is given."""
        dev, S = self.device, sl.S
        scr = torch.empty(S * (LANES * 4 + 3) + 2 * n_groups, dtype=torch.float32, device=dev)
        stats = scr[:S * LANES * 4]
        slot_sums = scr[S * LANES * 4:S * (LANES * 4 + 3)]
        out = scr[S * (LANES * 4 + 3):].view(2, n_groups)
        ans, _keep = self.dg.answers["hr2o"]
        _lib.check(_L().rl_cells_softmax_ce(
            self.dg.ref(), sl.ref(), C.byref(sl.cells), C.byref(ans), float(smoothing), _ptr(bias), self.acc.data_ptr(),
            zc.data_ptr(), int(n_groups), _ptr(group_ptr), float(grad_scale), stats.data_ptr(),
            slot_sums.data_ptr(), out[0].data_ptr(), out[1].data_ptr(), _ptr(Gc), _ptr(grad_bias), _stream()),
            "rl_cells_softmax_ce")
        return out[0], out[1]

    def predictor_backward(self, sl, Gc, grad_w):
        _lib.check(_L().rl_predictor_item_backward(self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), C.byref(sl.cells),
                                                  Gc.data_ptr(), grad_w.data_ptr(), _stream()), "rl_predictor_item_backward")

    def rank(self, sl, bias, sorted_bias, zc, which):
        counters = torch.empty(sl.S * 64, dtype=torch.int32, device=self.device)
        LH = torch.empty(sl.S * LANES, 2, dtype=torch.int64, device=self.device)
        known, _keep = self.dg.answers[which]
        _lib.check(_L().rl_cells_rank(self.dg.ref(), sl.ref(), C.byref(sl.cells), C.byref(known), _ptr(bias),
                                      _ptr(sorted_bias), zc.data_ptr(), counters.data_ptr(), LH.data_ptr(), _stream()),
                   "rl_cells_rank")
        return LH

    def add_to_dense(self, sl, zc, Z):
        _lib.check(_L().rl_cells_add_to_dense(self.dg.ref(), sl.ref(), C.byref(sl.cells), zc.data_ptr(), Z.data_ptr(),
                                              _stream()), "rl_cells_add_to_dense")

    def gather_dense(self, sl, G, Gc):
        _lib.check(_L().rl_cells_gather_dense(self.dg.ref(), sl.ref(), C.byref(sl.cells), G.data_ptr(), Gc.data_ptr(),
                                              _stream()), "rl_cells_gather_dense")

    def plus_features(self, sl, emb, F):
        _lib.check(_L().rl_plus_item_features(self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), C.byref(sl.cells),
                                             emb.data_ptr(), 16, F.data_ptr(), _stream()), "rl_plus_item_features")

    def plus_backward(self, sl, dF, grad_emb):
        _lib.check(_L().rl_plus_item_backward(self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), C.byref(sl.cells), 16,
                                             dF.data_ptr(), grad_emb.data_ptr(), _stream()), "rl_plus_item_backward")

    def tail_forward(self, sl, F, wts, zc, bits, front_done=False):
        _lib.check(_L().rl_tail_forward(C.byref(sl.cells), sl.slot_head.data_ptr(), 16, 128, F.data_ptr(),
                                        *[t.data_ptr() for t in wts], zc.data_ptr(), bits.data_ptr(),
                                        int(front_done), _stream()), "rl_tail_forward")

    def tail_backward(self, sl, R, F, wts, Gc, bits, dF, dY, grads, scratch, front_done=False):
        _lib.check(_L().rl_tail_backward(C.byref(sl.cells), sl.slot_head.data_ptr(), int(R), 16, 128, F.data_ptr(),
                                         *[t.data_ptr() for t in wts], Gc.data_ptr(), bits.data_ptr(),
                                         dF.data_ptr(), dY.data_ptr(), *[t.data_ptr() for t in grads], scratch.data_ptr(),
                                         int(front_done), _stream()), "rl_tail_backward")

    # ---- PNA aggregator (rl_pna.cu) ----
    def pna_stats(self, sl, emb, pna):
        _lib.check(_L().rl_pna_item_stats(self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), C.byref(sl.cells), emb.data_ptr(),
                                          C.byref(pna), _stream()), "rl_pna_item_stats")

    def pna_front_forward(self, sl, pna, W, b, Y, FEAT, SC):
        qscr = torch.empty(2 * sl.S * LANES, dtype=torch.float32, device=self.device)
        _lib.check(_L().rl_pna_front_forward(sl.ref(), C.byref(sl.cells), C.byref(pna), W.data_ptr(), b.data_ptr(), qscr.data_ptr(),
                                             Y.data_ptr(), FEAT.data_ptr(), SC.data_ptr(), _stream()), "rl_pna_front_forward")

    def pna_front_backward(self, sl, pna, W, dY, FEAT, SC, dstat, gW):
        _lib.check(_L().rl_pna_front_backward(C.byref(sl.cells), C.byref(pna), W.data_ptr(), dY.data_ptr(), FEAT.data_ptr(),
                                              SC.data_ptr(), dstat.data_ptr(), gW.data_ptr(), _stream()), "rl_pna_front_backward")

    def pna_backward(self, sl, emb, pna, dstat, grad_emb):
        _lib.check(_L().rl_pna_item_backward(self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), C.byref(sl.cells), emb.data_ptr(),
                                             C.byref(pna), dstat.data_ptr(), grad_emb.data_ptr(), _stream()), "rl_pna_item_backward")


def cell_kernels(sk) -> CellKernels:
    ck = getattr(sk, "_cells", None)
    if ck is None:
        ck = sk._cells = CellKernels(sk)
    return ck


# ================================================================================================
# Predictor (src/predictors.py:17-80)
# ================================================================================================
def predictor_step(model, sk, sl, smoothing, grad_scale, gw, gb, expanded=False, bits=32):
    """Enqueue ground -> cells -> scores -> CE -> backward for prepared slots; no host sync.
    gw / gb: zeroed gradient tensors (gb None without a bias).  -> (loss[ng], tsum[ng]) device tensors."""
    ck = cell_kernels(sk)
    if not expanded:
        sk.gr._run(sl, bits)
    _, (zc, Gc) = sk.gr.build_cells(sl, 2)
    bias = model.bias.detach() if model.entity_feature == "bias" else None
    if bias is not None:
        ck.bias_stats(bias)
    ck.predictor_scores(sl, model.rule_weights.detach(), zc)          # also leaves the non-zero counts in coordinate form
    loss, tsum = ck.softmax_ce(sl, bias, zc, smoothing, sl.group_ptr_dev, len(sl.group_sizes), grad_scale, Gc, gb)
    ck.predictor_backward(sl, Gc, gw)
    return loss, tsum


@torch.no_grad()
def predictor_rank(model, sk, sl, split, bits=32, expanded=False):
    """(L,H) int64[S*32,2] of prepared eval slots (trainer.py:173,189-201)."""
    ck = cell_kernels(sk)
    if not expanded:
        sk.gr.ground(sl)
    _, (zc,) = sk.gr.build_cells(sl, 1)
    bias = model.bias.detach() if model.entity_feature == "bias" else None
    ck.predictor_scores(sl, model.rule_weights.detach(), zc)
    sorted_bias = torch.sort(bias)[0] if bias is not None else None
    return ck.rank(sl, bias, sorted_bias, zc, "hr2oo" if split == "valid" else "hr2ooo")


# ================================================================================================
# PredictorPlus with the sum aggregator, hidden_dim 16, MLP(2H,[128,1]) (every shipped config but WN18RR's pna)
# ================================================================================================
def plus_cells_supported(model) -> bool:
    sm = model.score_model
    return (model.aggregator in ("sum", "pna") and model.hidden_dim == 16 and len(sm.layers) == 2
            and sm.layers[0].out_features == 128 and sm.layers[1].out_features == 1 and sm.batch_norms is None
            and not sm.short_cut and sm.dropout is None)


PLUS_PLANES = 2 + 4 * 16 + 4          # zc, Gc | F, dF, O, dY [16 each] | ReLU bits [4 words]
PNA_PLANES = PLUS_PLANES + 16 + 16 + 32 + 32 + 64 + 64 + 2    # + s1, s2 | min keys, max keys (u64 x 16) | FEAT | dstat | deg, SC


def _plus_planes(planes, pna=False):
    """Per-cell arrays of the PredictorPlus step in the planes of build_cells (contiguous [cap][16] blocks)."""
    blk = lambda i0, n: planes[i0:i0 + n].view(-1)
    pl = {"zc": blk(0, 1), "Gc": blk(1, 1), "F": blk(2, 16), "dF": blk(18, 16), "O": blk(34, 16), "dY": blk(50, 16),
          "bits": blk(66, 4)}
    if pna:
        pl.update({"s1": blk(70, 16), "s2": blk(86, 16), "mnk": blk(102, 32), "mxk": blk(134, 32), "FEAT": blk(166, 64),
                   "dstat": blk(230, 64), "deg": blk(294, 1), "SC": blk(295, 1)})
        pl["pna"] = _lib.RlPna(pl["s1"].data_ptr(), pl["s2"].data_ptr(), pl["deg"].data_ptr(), pl["mnk"].data_ptr(),
                               pl["mxk"].data_ptr())
    return pl


def _tail_weights(model):
    r2e, sm = model.rule_to_entity, model.score_model
    lin0 = r2e.add_model.layers[0]
    return [lin0.weight, lin0.bias, r2e.layer_norm.weight, r2e.layer_norm.bias, sm.layers[0].weight, sm.layers[0].bias,
            sm.layers[1].weight, sm.layers[1].bias, model.relation_emb.weight]


def _step_rule_ids(model, sl, device):
    """Global ids of the rules of the heads present in this call (host-known: no sync)."""
    heads = np.unique(sl.heads)
    if len(heads) == 1:                                                 # one-batch steps (and their CUDA graphs): device-resident per head
        cache = model.__dict__.setdefault("_head_rule_ids", {})
        key = (int(heads[0]), str(device))
        if key not in cache:
            cache[key] = torch.from_numpy(model.compiled.head_rule_array[key[0]]).to(device)
        return cache[key]
    ids = np.concatenate([model.compiled.head_rule_array[int(q)] for q in heads]) if len(heads) else np.zeros(0, np.int64)
    return torch.from_numpy(ids).to(device, non_blocking=True)


def _encode_rules(model, ids):
    """Output of the rule encoder (rnn / lstm / gru) for the rules ``ids``, with autograd when it is enabled."""
    if model.rule_features.device != ids.device:
        model.rule_features = model.rule_features.to(ids.device)
    return model.encode_rules(model.rule_features[ids])


def _rule_embeddings(model, sl, device):
    """-> (emb [num_rules,16] fp32 indexed by global rule id, (ids, encoder output) or None)."""
    if model.type == "emb":
        return model.rule_emb.detach(), None
    ids = _step_rule_ids(model, sl, device)
    full = model._emb_scratch(device)
    if ids.numel() == 0:
        return full, None
    with torch.enable_grad():
        sub = _encode_rules(model, ids)                                       # rule encoder: small autograd graph
    full.index_copy_(0, ids, sub.detach().float())
    return full, (ids, sub)


def _plus_scores(model, ck, sl, pl, emb, wts):
    """Forward half of a PredictorPlus step on the cells: aggregate the rule embeddings ``emb`` (sum, or the PNA
    statistics + front) -> dense tail -> pl["zc"]."""
    pna = model.aggregator == "pna"
    if pna:                                                              # statistics -> scalers + Linear(12H,H) -> F holds y
        ck.pna_stats(sl, emb, pl["pna"])
        ck.pna_front_forward(sl, pl["pna"], wts[0], wts[1], pl["F"], pl["FEAT"], pl["SC"])
    else:
        ck.plus_features(sl, emb, pl["F"])
    ck.tail_forward(sl, pl["F"], wts, pl["zc"], pl["bits"], front_done=pna)


def _plus_backward(model, ck, sl, pl, emb, wts, grads, grad_emb):
    """Backward half: pl["Gc"] -> dense tail -> aggregate.  ACCUMULATES into ``grads`` (the _tail_weights) and
    ``grad_emb`` [num_rules,16] (None: the step has no rule to take a gradient)."""
    pna = model.aggregator == "pna"
    ck.tail_backward(sl, model.num_relations, pl["F"], wts, pl["Gc"], pl["bits"], pl["dF"], pl["dY"], grads,
                     model._d1sum_scratch(ck.device), front_done=pna)
    if grad_emb is None:
        return
    if pna:
        ck.pna_front_backward(sl, pl["pna"], wts[0], pl["dY"], pl["FEAT"], pl["SC"], pl["dstat"], grads[0])
        ck.pna_backward(sl, emb, pl["pna"], pl["dstat"], grad_emb)
    else:
        ck.plus_backward(sl, pl["dF"], grad_emb)


def plus_step(model, sk, sl, smoothing, grad_scale, gbuf: GradBuffer, expanded=False, bits=32, want_grad=True):
    """ground -> cells -> aggregate -> fused tail -> CE -> hand-written backward into every parameter of
    PredictorPlus (gradients accumulate into ``gbuf``'s views, zeroed by the caller).  No host sync.
    -> (loss[ng], tsum[ng]) device tensors."""
    ck = cell_kernels(sk)
    dev = sk.device
    if not expanded:
        sk.gr._run(sl, bits)
    pna = model.aggregator == "pna"
    _, planes = sk.gr.build_cells(sl, PNA_PLANES if pna else PLUS_PLANES)
    pl = _plus_planes(planes, pna)
    zc, Gc = pl["zc"], pl["Gc"]
    emb, enc = _rule_embeddings(model, sl, dev)
    wts = [t.detach() for t in _tail_weights(model)]
    _plus_scores(model, ck, sl, pl, emb, wts)
    ef = model.entity_feature
    ng = len(sl.group_sizes)
    extra = None
    if ef == "RotatE":
        with torch.enable_grad():
            extra = model.RotatE.slot_scores(sk, sl)                               # dense by nature: [S][N][32]
        Z = extra.detach()
        ck.add_to_dense(sl, zc, Z)
        loss, tsum, G = sk.softmax_ce(sl, Z, sl.nzmask, smoothing, False, sl.group_ptr_dev, ng, want_grad=want_grad)
        if want_grad:
            if grad_scale != 1.0:
                G.mul_(grad_scale)
            ck.gather_dense(sl, G, Gc)
    else:
        bias = model.bias.detach() if ef == "bias" else None
        if bias is not None:
            ck.bias_stats(bias)
        loss, tsum = ck.softmax_ce(sl, bias, zc, smoothing, sl.group_ptr_dev, ng, grad_scale, Gc if want_grad else None,
                                   gbuf.view(model.bias) if (bias is not None and want_grad) else None)
    if not want_grad:
        return loss, tsum
    grads = [gbuf.view(p) for p in _tail_weights(model)]
    if model.type == "emb":
        gemb = gbuf.view(model.rule_emb)
    else:
        gemb = model._emb_scratch(dev, grad=True).zero_() if enc is not None else None
    _plus_backward(model, ck, sl, pl, emb, wts, grads, gemb)
    if enc is not None:
        ids, sub = enc
        enc_params = [model.vocab_emb.weight] + [p for p in model.rnn.parameters()]
        gs = torch.autograd.grad(sub, enc_params, gemb[ids].to(sub.dtype), allow_unused=True)
        for p, g_ in zip(enc_params, gs):
            if g_ is not None:
                gbuf.view(p).add_(g_)
    if extra is not None:
        rp = [model.RotatE.eemb, model.RotatE.remb]
        gs = torch.autograd.grad(extra, rp, G, allow_unused=True)
        for p, g_ in zip(rp, gs):
            if g_ is not None:
                gbuf.view(p).add_(g_)
    return loss, tsum


@torch.no_grad()
def plus_rank(model, sk, sl, split):
    ck = cell_kernels(sk)
    dev = sk.device
    sk.gr.ground(sl)
    pna = model.aggregator == "pna"
    _, planes = sk.gr.build_cells(sl, PNA_PLANES if pna else PLUS_PLANES)
    pl = _plus_planes(planes, pna)
    zc = pl["zc"]
    emb, _ = _rule_embeddings(model, sl, dev)
    _plus_scores(model, ck, sl, pl, emb, [t.detach() for t in _tail_weights(model)])
    which = "hr2oo" if split == "valid" else "hr2ooo"
    ef = model.entity_feature
    if ef == "RotatE":
        Z = model.RotatE.slot_scores(sk, sl).detach()
        ck.add_to_dense(sl, zc, Z)
        return sk.filtered_rank(sl, Z, sl.nzmask, which, False)
    bias = model.bias.detach() if ef == "bias" else None
    sorted_bias = torch.sort(bias)[0] if bias is not None else None
    return ck.rank(sl, bias, sorted_bias, zc, which)


# ================================================================================================
# The reference's forward(all_h, all_r, edges_to_remove) -> (score [B,N], mask [B,N]) on the cells.  Two calls may be
# alive before one backward(), so nothing here lives in the workspaces the fused steps reuse: the slots, the cell
# arrays, the rule-embedding table and the gradients all belong to the call.
# ================================================================================================
def call_cells(sk, sl, floats_per_cell):
    """rl_cells_build for a grounded API call into arrays of its own -> (planes, number of cells).  When the cells do
    not fit, the frontier is expanded again and the cells built with exactly the count k_cell_scan reported."""
    _, planes = sk.gr.build_cells(sl, floats_per_cell, cap=sk.gr.cell_capacity(sl))
    n, over = sl.cell_counters[:2].tolist()
    if over:
        sk.gr._run(sl, sl.count_bits)
        _, planes = sk.gr.build_cells(sl, floats_per_cell, cap=n)
    return planes, n


class _CellScoresFn(torch.autograd.Function):
    """Cell scores of a Predictor (params: rule_weights) or a PredictorPlus (params: rule_emb or the encoder output of
    the rules ``ids``, then the _tail_weights; none when the call has no cell) -> the reference's score [B,N]:
    bias[e] (or the RotatE logits, or 0) + the cell's score, -inf outside the cells without an entity feature."""

    @staticmethod
    def forward(ctx, model, sk, sl, planes, ids, bias, extra, *params):
        ck = cell_kernels(sk)
        S, N = sl.S, sk.N
        if extra is not None:
            Z = extra.detach().clone()
        elif bias is not None:
            Z = bias.detach().view(1, N, 1).expand(S, N, LANES).contiguous()
        else:
            Z = torch.zeros(S, N, LANES, dtype=torch.float32, device=sk.device)
        plus = hasattr(model, "score_model")
        emb = wts = pl = None
        if not plus:
            ck.predictor_scores(sl, params[0].detach(), planes[0])
            zc = planes[0]
        elif params:
            pl = _plus_planes(planes, model.aggregator == "pna")
            emb = params[0].detach()
            if ids is not None:                                          # encoder output -> table indexed by global rule id
                emb = torch.zeros(model.num_rules, model.hidden_dim, dtype=torch.float32, device=sk.device).index_copy_(
                    0, ids, emb.float())
            wts = [t.detach() for t in params[1:]]
            _plus_scores(model, ck, sl, pl, emb, wts)
            zc = pl["zc"]
        if not plus or params:
            ck.add_to_dense(sl, zc, Z)
        score, nz = sk.to_dense(sl, Z, sl.nzmask)
        if bias is None and extra is None:
            score.masked_fill_(~nz, float("-inf"))
        ctx.model, ctx.sk, ctx.sl, ctx.planes, ctx.ids, ctx.pl, ctx.emb, ctx.wts = model, sk, sl, planes, ids, pl, emb, wts
        ctx.has_bias, ctx.has_extra, ctx.params = bias is not None, extra is not None, [p.detach() for p in params]
        ctx.mark_non_differentiable(nz)
        return score, nz

    @staticmethod
    def backward(ctx, gscore, _gnz):
        model, sk, sl, params = ctx.model, ctx.sk, ctx.sl, ctx.params
        ck = cell_kernels(sk)
        G = sk.from_dense(sl, gscore.contiguous())
        grads = ()
        if ctx.pl is None and params:                                    # Predictor
            ck.gather_dense(sl, G, ctx.planes[1])
            gw = torch.zeros_like(params[0])
            ck.predictor_backward(sl, ctx.planes[1], gw)
            grads = (gw,)
        elif params:
            ck.gather_dense(sl, G, ctx.pl["Gc"])
            gt = [torch.zeros_like(p) for p in params[1:]]
            gemb = torch.zeros_like(ctx.emb)
            _plus_backward(model, ck, sl, ctx.pl, ctx.emb, ctx.wts, gt, gemb)
            grads = (gemb if ctx.ids is None else gemb[ctx.ids].to(params[0].dtype),) + tuple(gt)
        gb = G.sum(dim=(0, 2)) if ctx.has_bias else None
        return (None, None, None, None, None, gb, G if ctx.has_extra else None) + grads


def predictor_api_scores(model, sk, sl):
    """Predictor.forward on a grounded call -> (score [B,N], nonzero mask [B,N], number of cells)."""
    planes, n = call_cells(sk, sl, 2)                                    # zc, Gc
    bias = model.bias if model.entity_feature == "bias" else None
    score, nz = _CellScoresFn.apply(model, sk, sl, planes, None, bias, None, model.rule_weights)
    return score, nz, n


def plus_api_scores(model, sk, sl):
    """PredictorPlus.forward on a grounded call (plus_cells_supported(model)) -> (score, nonzero mask, number of
    cells).  Without a cell only the entity feature takes part (predictors.py:230-237)."""
    planes, n = call_cells(sk, sl, PNA_PLANES if model.aggregator == "pna" else PLUS_PLANES)
    ef = model.entity_feature
    bias = model.bias if ef == "bias" else None
    extra = model.RotatE.slot_scores(sk, sl) if ef == "RotatE" else None
    ids, params = None, ()
    if n > 0:
        if model.type == "emb":
            params = (model.rule_emb,) + tuple(_tail_weights(model))
        else:
            ids = _step_rule_ids(model, sl, sk.device)
            params = (_encode_rules(model, ids),) + tuple(_tail_weights(model))
    score, nz = _CellScoresFn.apply(model, sk, sl, planes, ids, bias, extra, *params)
    return score, nz, n


# ================================================================================================
# The reference's own schedule -- ONE batch of <= 32 queries per optimizer step (src/trainer.py:68-95) -- is launch
# bound: ~25 small kernels, a memset, two copies and the Python around them per 32 queries.  Every size of such a
# step depends only on the batch's head relation, so the whole step (H2D of the queries -> slot preparation ->
# expansion -> cells -> scores -> CE -> backward -> D2H of loss / flags) is captured ONCE per head relation as a CUDA
# graph and replayed with new queries written into its pinned staging buffer.
# ================================================================================================
class GraphTrainStep:
    """Captured fused train step of ``model`` for batches of one head relation (one slot), as TWO CUDA graphs:

      ground  H2D of the queries -> slot preparation -> frontier expansion          (independent of the parameters)
      score   cells -> scores -> CE -> backward -> D2H of loss / counts / flags     (reads the current parameters)

    so a trainer can enqueue the grounding of step k+1 behind the scoring of step k and only then wait for step k's
    result: the GPU expands the next frontier while the host reads the loss, exchanges gradients and steps the optimizer."""

    def __init__(self, model, head: int, smoothing: float):
        from .engine import HostStep, Slots
        self.model, self.head, self.smoothing = model, int(head), float(smoothing)
        dev = next(model.parameters()).device
        self.sk = sk = model._driver(dev)
        gr = sk.gr
        self.params = model.fused_params()
        # static host staging: 32 query columns (padding = -1), rows h, t
        q = np.full((2, LANES), -1, dtype=np.int64)
        self.host = HostStep(gr.cr, np.array([self.head], dtype=np.int64), np.array([0, 0], dtype=np.int64), host_queries=q,
                             group_sizes=[0], remove_query_edges=True)
        self._pack = self.host.staged.numpy()
        self._q = self._pack[:2 * LANES].reshape(2, LANES)
        self._qoff = self._pack[self.host.n64:].view(np.int32)[1:3]           # q_off = [0, n] behind the slot head
        self.generation = gr.generation

        def ground():
            sl = Slots(gr.dg, self.host)
            sl.use_workspace, sl.coo_only = True, True
            gr._run(sl, 32)
            return sl

        def score(sl):
            gbuf = GradBuffer(self.params)
            loss, tsum = model.step_on_slots(sk, sl, self.smoothing, 1.0, gbuf, 32, expanded=True)
            pack = torch.cat([loss, tsum, sl.slot_ncell.float(), sl.flags.float()])
            return gbuf, pack

        self._fill(np.zeros((1, 3), dtype=np.int64) + np.array([[0, self.head, 0]]))
        _, pack = score(ground())                                            # eager warm-up: sizes every workspace
        self.pinned = torch.empty(pack.numel(), dtype=torch.float32, pin_memory=True)
        torch.cuda.synchronize()
        self.generation = gr.generation
        self.g_ground, self.g_score = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_ground):
            self.sl = ground()
        with torch.cuda.graph(self.g_score, pool=self.g_ground.pool()):
            self.gbuf, pack = score(self.sl)
            self.pinned.copy_(pack, non_blocking=True)
        if gr.generation != self.generation:
            raise _lib.RlError("a workspace was reallocated during graph capture")
        self.ev_in, self.ev_out = torch.cuda.Event(), torch.cuda.Event()
        self._in_flight = False

    def _fill(self, batch: np.ndarray):
        n = int(batch.shape[0])
        self._q[:, :] = -1
        self._q[0, :n] = batch[:, 0]
        self._q[1, :n] = batch[:, 2]
        self._qoff[0], self._qoff[1] = 0, n
        self.n = n

    def launch_ground(self, batch: np.ndarray):
        """Enqueue the parameter-independent half for ``batch`` [n,3] (no host wait unless this head's previous
        queries are still being copied)."""
        if self._in_flight:
            self.ev_in.synchronize()                                         # the staging buffer is read by the graph's H2D node
        self._fill(batch)
        self.g_ground.replay()
        self.ev_in.record()
        self._in_flight = True

    def launch_score(self):
        self.g_score.replay()
        self.ev_out.record()

    def result(self):
        """-> (loss, target_sum, cells, flags) of the last launch_score, after waiting for it; gradients are in self.gbuf."""
        self.ev_out.synchronize()
        host = self.pinned
        return float(host[0]), float(host[1]), int(host[2]), host[3:]

    def __call__(self, batch: np.ndarray):
        self.launch_ground(batch)
        self.launch_score()
        return self.result()


def graph_step_for(model, batch, smoothing: float):
    """The captured step of the batch's head relation (captured on first use), or None when the step has to take the
    eager path (more than 32 queries, unsupported model, capture not possible)."""
    if len(batch) > LANES or not getattr(model, "supports_pipeline", False) or model.__dict__.get("_graphs_broken", False):
        return None
    head = int(batch[0][1])
    cache = model.__dict__.setdefault("_graph_steps", {})
    gs = cache.get((head, float(smoothing)))
    gr = model._driver(next(model.parameters()).device).gr
    if gs is None or gs.generation != gr.generation:
        gr.reserve_single_slot()
        try:
            gs = cache[(head, float(smoothing))] = GraphTrainStep(model, head, smoothing)
        except _lib.RlError:
            raise
        except RuntimeError as e:                                            # an op of this model cannot be captured: eager from now on
            import logging
            logging.warning("per-head CUDA graphs disabled for this model: %s", str(e).splitlines()[0])
            model.__dict__["_graphs_broken"] = True
            torch.cuda.synchronize()
            return None
    return gs


def graph_step_result(model, gs: GraphTrainStep):
    """(loss, tsum, cells, gbuf) of a launched step, or None when it has to be redone eagerly (count overflow, cell
    arrays too small)."""
    loss, tsum, cells, flags = gs.result()
    if flags[8] != 0 or flags[1] != 0:
        gs.sk.gr.note_cell_count(cells)
        return None
    return loss, tsum, cells, gs.gbuf


def graph_train_step(model, batch: np.ndarray, smoothing: float):
    """One reference-schedule train step through the per-head CUDA graphs, synchronously.  Returns (loss, tsum, cells,
    gbuf) or None when the step has to take the eager path."""
    batch = np.asarray(batch, dtype=np.int64).reshape(-1, 3)
    gs = graph_step_for(model, batch, smoothing)
    if gs is None:
        return None
    gs.launch_ground(batch)
    gs.launch_score()
    return graph_step_result(model, gs)
