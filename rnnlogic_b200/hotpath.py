"""Kernel drivers for the scoring half of the hot path: rule-weight aggregation, softmax-CE with
its backward, filtered rank and metrics (kernels (2) and (3) of include/rnnlogic_b200.h).

Everything here works on entity-major per-slot matrices [S][N][32]; ``to_dense`` converts to the
reference's [B,N] layout when the Python API has to return it."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from .engine import Grounder, Slots, _stream

LANES = _lib.LANES


class ScoreKernels:
    def __init__(self, grounder: Grounder):
        self.gr = grounder
        self.dg, self.dr, self.cr = grounder.dg, grounder.dr, grounder.cr
        self.N = grounder.graph.entity_size
        self.device = grounder.device
        self.nblk = _lib.lib().rl_softmax_blocks(self.N)
        self._scales = {}

    def slot_scale(self, S: int, value: float) -> Optional[torch.Tensor]:
        """float32[S] filled with ``value`` (None for 1.0); cached -- the same few shapes recur every step."""
        if value == 1.0:
            return None
        key = (int(S), float(value))
        t = self._scales.get(key)
        if t is None:
            if len(self._scales) > 64:
                self._scales.clear()
            t = self._scales[key] = torch.full((S,), float(value), dtype=torch.float32, device=self.device)
        return t

    # ---- kernel (2a) -------------------------------------------------------------------------
    def predictor_scores(self, sl: Slots, w: torch.Tensor, bias: Optional[torch.Tensor], fill_neg_inf: bool,
                         partial: Optional[torch.Tensor] = None):
        """partial (S*nblk*64 floats): also leave the softmax partials of every query there."""
        Z = torch.empty(sl.S, self.N, LANES, dtype=torch.float32, device=self.device)
        nzmask = torch.empty(sl.S, self.N, dtype=torch.int32, device=self.device)
        _lib.check(_lib.lib().rl_predictor_scores(
            self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), w.data_ptr(),
            bias.data_ptr() if bias is not None else None, int(fill_neg_inf), Z.data_ptr(), nzmask.data_ptr(),
            partial.data_ptr() if partial is not None else None, _stream()), "rl_predictor_scores")
        return Z, nzmask

    def predictor_train_tail(self, sl: Slots, w, bias, smoothing: float, group_ptr, n_groups: int,
                             slot_scale: Optional[torch.Tensor], grad_w, grad_bias):
        """aggregate -> CE -> backward of Predictor with the passes fused (rl_predictor_scores with
        softmax partials + rl_predictor_ce_backward).  -> (group_loss, group_tsum, nzmask)."""
        dev, S = self.device, sl.S
        use_mask = bias is None
        partial = torch.empty(S * self.nblk * 64, dtype=torch.float32, device=dev)
        Z, nzmask = self.predictor_scores(sl, w, bias, use_mask, partial)
        stats = torch.empty(S * LANES * 4, dtype=torch.float32, device=dev)
        slot_sums = torch.empty(3 * S, dtype=torch.float32, device=dev)
        out = torch.empty(2, n_groups, dtype=torch.float32, device=dev)
        ans, _keep = self.dg.answers["hr2o"]
        G = torch.empty_like(Z)                                   # gradient rows: held until the call is enqueued
        _lib.check(_lib.lib().rl_predictor_ce_backward(
            self.dg.ref(), self.dr.ref(), sl.ref(), sl.fref(), C.byref(ans), float(smoothing), int(use_mask),
            Z.data_ptr(), nzmask.data_ptr(), int(n_groups), group_ptr.data_ptr() if group_ptr is not None else None,
            partial.data_ptr(), 1, stats.data_ptr(), slot_sums.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
            G.data_ptr(), slot_scale.data_ptr() if slot_scale is not None else None, grad_w.data_ptr(),
            grad_bias.data_ptr() if grad_bias is not None else None, _stream()), "rl_predictor_ce_backward")
        return out[0], out[1], nzmask

    # ---- kernel (2b) -------------------------------------------------------------------------
    def softmax_ce(self, sl: Slots, Z, nzmask, smoothing: float, use_mask: bool,
                   group_ptr: Optional[torch.Tensor], n_groups: int, want_grad: bool = True):
        """-> (group_loss[n_groups], group_tsum[n_groups], G[S][N][32] | None)."""
        dev = self.device
        S = sl.S
        partial = torch.empty(S * self.nblk * 64, dtype=torch.float32, device=dev)
        stats = torch.empty(S * LANES * 4, dtype=torch.float32, device=dev)
        slot_sums = torch.empty(3 * S, dtype=torch.float32, device=dev)
        out = torch.empty(2, n_groups, dtype=torch.float32, device=dev)
        G = torch.empty_like(Z) if want_grad else None
        ans, _keep = self.dg.answers["hr2o"]
        _lib.check(_lib.lib().rl_softmax_ce(
            self.dg.ref(), sl.ref(), C.byref(ans), float(smoothing), int(use_mask), Z.data_ptr(), nzmask.data_ptr(),
            int(n_groups), group_ptr.data_ptr() if group_ptr is not None else None, partial.data_ptr(),
            stats.data_ptr(), slot_sums.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
            G.data_ptr() if G is not None else None, _stream()), "rl_softmax_ce")
        return out[0], out[1], G

    # ---- kernel (3) --------------------------------------------------------------------------
    def filtered_rank(self, sl: Slots, Z, nzmask, which: str, use_mask: bool) -> torch.Tensor:
        """int64[S*32, 2] (L,H) per lane (0,0 on padding lanes); which = 'hr2oo' | 'hr2ooo'."""
        counters = torch.empty(sl.S * 64, dtype=torch.int32, device=self.device)
        LH = torch.empty(sl.S * LANES, 2, dtype=torch.int64, device=self.device)
        known, _keep = self.dg.answers[which]
        _lib.check(_lib.lib().rl_filtered_rank(
            self.dg.ref(), sl.ref(), C.byref(known), int(use_mask), Z.data_ptr(), nzmask.data_ptr(),
            counters.data_ptr(), LH.data_ptr(), _stream()), "rl_filtered_rank")
        return LH

    def rank_metrics(self, LH: torch.Tensor, weight: Optional[torch.Tensor], expectation: bool) -> torch.Tensor:
        """fp64[5] partial sums (hit1, hit3, hit10, mr, mrr) over the rows of LH."""
        sums = torch.zeros(5, dtype=torch.float64, device=self.device)
        LH = LH.contiguous()
        _lib.check(_lib.lib().rl_rank_metrics(
            int(LH.shape[0]), LH.data_ptr(), weight.data_ptr() if weight is not None else None, int(expectation),
            self.dg.harmonic.data_ptr(), sums.data_ptr(), _stream()), "rl_rank_metrics")
        return sums

    # ---- layout conversion --------------------------------------------------------------------
    def to_dense(self, sl: Slots, Z, nzmask):
        """(score fp32[Q,N], nonzero bool[Q,N]) in the reference's layout."""
        Q = int(sl.q_off[-1])
        score = torch.empty(Q, self.N, dtype=torch.float32, device=self.device)
        mask = torch.empty(Q, self.N, dtype=torch.uint8, device=self.device)
        L = _lib.lib()
        for s in range(sl.S):
            q0, nq = int(sl.q_off[s]), int(sl.nq[s])
            _lib.check(L.rl_slot_to_dense(self.N, nq, Z[s].data_ptr(), score[q0].data_ptr(), self.N, _stream()))
            _lib.check(L.rl_mask_to_dense(self.N, nq, nzmask[s].data_ptr(), mask[q0].data_ptr(), self.N, _stream()))
        return score, mask.bool()

    def from_dense(self, sl: Slots, dense: torch.Tensor) -> torch.Tensor:
        """fp32[Q,N] -> entity-major [S][N][32] (zero padding lanes)."""
        out = torch.zeros(sl.S, self.N, LANES, dtype=torch.float32, device=self.device)
        for s in range(sl.S):
            q0, nq = int(sl.q_off[s]), int(sl.nq[s])
            out[s, :, :nq] = dense[q0:q0 + nq].t()
        return out


def dense_filtered_rank(logits: torch.Tensor, flag: torch.Tensor, mask: torch.Tensor, all_t: torch.Tensor):
    """(L,H) int64[Q,2] from the reference's dense tensors (trainer.py:189-201)."""
    for name, t in (("logits", logits), ("flag", flag), ("mask", mask), ("all_t", all_t)):
        _lib.require_cuda(t, name)
    Q, N = logits.shape
    lg = logits.detach().contiguous().float()
    fl = flag.contiguous().to(torch.uint8)
    mk = mask.contiguous().to(torch.uint8)
    tt = all_t.contiguous().to(torch.int64)
    LH = torch.empty(Q, 2, dtype=torch.int64, device=logits.device)
    _lib.check(_lib.lib().rl_filtered_rank_dense(Q, N, lg.data_ptr(), fl.data_ptr(), mk.data_ptr(), tt.data_ptr(),
                                                 LH.data_ptr(), _stream()), "rl_filtered_rank_dense")
    return LH
