"""``GraphNet`` with the reference's constructor, ``forward`` and checkpoint API, scored by libgnnb on the GPU.

Mirrors graphnet/graph_conv.py of oval-group/GNN_branching: ``GraphNet(T, p)`` (:473-483) owns submodules named
``EmbedUpdates`` (:394-417, holding ``update`` = ``EmbedLayerUpdate`` :22-74) and ``ComputeFinalScore`` (:421-432),
so the 52 ``state_dict`` keys are identical and ``models/cifar_trained_gnn/*.pt`` loads unchanged.  The modules
only hold parameters; all arithmetic runs in the CUDA library.  There is no PyTorch / CPU fallback.
"""
from __future__ import annotations

from typing import List, Optional

import torch
from torch import nn

from .engine import Scorer
from .frontier import Frontier


class EmbedLayerUpdate(nn.Module):
    """Parameter holder with the reference's linears (graph_conv.py:26-74)."""

    def __init__(self, p, T):
        super().__init__()
        self.p, self.T = p, T
        self.inp_f = nn.Linear(3, p)
        self.inp_f_1 = nn.Linear(p, p)
        self.inp_b = nn.Linear(2, p)
        self.inp_b_1 = nn.Linear(p, p)
        self.inp_b2 = nn.Linear(2 * p, p)
        self.inp_b2_2 = nn.Linear(p, p)
        self.fc1 = nn.Linear(7, p)
        self.fc1_1 = nn.Linear(p, p)
        self.fc3 = nn.Linear(2 * p, p)
        self.fc3_2 = nn.Linear(p, p)
        self.fc4 = nn.Linear(2 * p, p)
        self.fc4_2 = nn.Linear(p, p)
        self.out1 = nn.Linear(4, p)
        self.out2 = nn.Linear(2 * p, p)
        self.out3 = nn.Linear(p, p)
        self.bc1 = nn.Linear(7, p)
        self.bc1_1 = nn.Linear(p, p)
        self.bc1_2 = nn.Linear(p, p)
        self.bc2 = nn.Linear(3 * p, p)
        self.bc2_1 = nn.Linear(p, p)
        self.bc3 = nn.Linear(2 * p, p)
        self.bc3_1 = nn.Linear(p, p)
        self.bc4 = nn.Linear(2 * p, p)
        self.bc4_1 = nn.Linear(p, p)


class EmbedUpdates(nn.Module):
    def __init__(self, T, p):
        super().__init__()
        self.T, self.p = T, p
        self.update = EmbedLayerUpdate(p, T)


class ComputeFinalScore(nn.Module):
    def __init__(self, p):
        super().__init__()
        self.p = p
        self.fnode = nn.Linear(p, p)
        self.fscore = nn.Linear(p, 1)


class GraphNet(nn.Module):
    """Drop-in for graphnet.graph_conv.GraphNet (graph_conv.py:473-483)."""

    def __init__(self, T, p, math: Optional[str] = None, chunk: int = 0, rescore: bool = False):
        super().__init__()
        if p != 64:
            raise NotImplementedError('the CUDA kernels are specialised for p = 64 (graph_score.py:9)')
        self.T, self.p = T, p
        self.EmbedUpdates = EmbedUpdates(T, p)
        self.ComputeFinalScore = ComputeFinalScore(p)
        self._math, self._chunk, self._rescore = math, chunk, rescore
        self._scorer: Optional[Scorer] = None

    # ---- engine plumbing ----
    def scorer(self, device_index: Optional[int] = None) -> Scorer:
        if device_index is None:
            q = next(self.parameters())
            device_index = q.device.index if q.device.type == 'cuda' else torch.cuda.current_device()
        if self._scorer is None or self._scorer.device != device_index:
            self._scorer = Scorer(device_index, math=self._math, chunk=self._chunk, rescore=self._rescore)
        key = tuple((q.data_ptr(), q._version) for q in self.parameters())
        if self._scorer._gnn_key != key:          # state_dict() costs ~0.2 ms: only when a parameter changed
            self._scorer.set_gnn(self.state_dict(), self.T, self.p, key=key)
        return self._scorer

    def adopt_weights(self, sc: Scorer) -> None:
        """After a device-side optimiser step: copy the context's parameters into this module (so ``state_dict()`` and
        checkpoints follow the fine-tuning) without triggering a re-upload."""
        new = sc.weights()
        with torch.no_grad():
            for k, q in self.state_dict().items():
                q.copy_(new[k])
        sc._gnn_key = tuple((q.data_ptr(), q._version) for q in self.parameters())

    def score_frontier(self, fr: Frontier, return_scores: bool = True):
        """Batched entry (addition to the reference API): (best_score [B], best_idx [B], scores [B, sum n_k])."""
        sc = self.scorer(fr.device.index if fr.device.type == 'cuda' else None)
        sc.set_network(fr.net, key=fr.net.key)
        return sc.score(fr, return_scores=return_scores)

    def score_frontier_topk(self, fr: Frontier, k: int, return_scores: bool = False):
        """The ``k`` best branching candidates of every subdomain (addition to the reference API): (top_score [B, k],
        top_idx [B, k], scores [B, sum n_k] or None); column 0 is ``score_frontier``'s decision."""
        sc = self.scorer(fr.device.index if fr.device.type == 'cuda' else None)
        sc.set_network(fr.net, key=fr.net.key)
        return sc.score_topk(fr, k, return_scores=return_scores)

    def forward(self, lower_bounds_all, upper_bounds_all, dual_vars, primals, primal_inputs, layers, masks) -> List[torch.Tensor]:
        """Same arguments and return value as the reference (graph_conv.py:479-483): a list with, per subdomain,
        the scores of the ReLUs whose mask entry is non-zero, in flat order.  Runs without autograd, as the
        reference's caller does (graph_score.py:32); the autograd variant is a later row (SURVEY §8f)."""
        fr = Frontier.from_reference_args(lower_bounds_all, upper_bounds_all, dual_vars, primals, primal_inputs,
                                          layers, masks)
        _, _, scores = self.score_frontier(fr, return_scores=True)
        return [scores[b][fr.mask[b].nonzero().view(-1)] for b in range(fr.B)]
