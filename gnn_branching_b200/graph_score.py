"""``GraphChoice`` with the reference's constructor and ``decision`` API (graphnet/graph_score.py:8-56)."""
from __future__ import annotations

import time

import torch

from .engine import flat_to_layer_index
from .frontier import Frontier
from .graph_conv import GraphNet


class GraphChoice:
    """Drop-in for graphnet.graph_score.GraphChoice.

    ``init_mask``: list of per-ReLU-layer int tensors in {-1, 0, 1}; ``model_name``: path of a GraphNet
    ``state_dict`` checkpoint (models/cifar_trained_gnn/*.pt loads unchanged).
    """
    verbose = False     # the reference prints 'graph requires: <s>' on every call (graph_score.py:36)

    def __init__(self, init_mask, model_name, linear=False, math=None, rescore=False):
        model = GraphNet(2, 64, math=math, rescore=rescore)         # graph_score.py:9
        model.load_state_dict(torch.load(model_name, map_location='cpu'))
        model.eval()
        self.model = model.cuda()
        trans_len, temp = [], 0
        for i in init_mask:                                          # graph_score.py:14-19
            temp += len(i)
            trans_len.append(temp)
        self.trans_len = torch.tensor(trans_len)
        self.hidden_sizes = [len(i) for i in init_mask]

    def decision(self, lower_bounds_all, upper_bounds_all, dual_vars, primal_input, primals, layers, mask):
        """-> [dec_lay, dec_idx].  Note the (primal_input, primals) order, swapped w.r.t. GraphNet.forward
        (graph_score.py:21 vs graph_conv.py:479)."""
        return self._decide(lower_bounds_all, upper_bounds_all, dual_vars, primal_input, primals, layers, mask, None)[0]

    def decision_topk(self, lower_bounds_all, upper_bounds_all, dual_vars, primal_input, primals, layers, mask, k):
        """-> up to ``k`` [dec_lay, dec_idx] pairs, best first (addition to the reference API); the first is ``decision``'s,
        there are min(k, undecided ReLUs) of them."""
        return self._decide(lower_bounds_all, upper_bounds_all, dual_vars, primal_input, primals, layers, mask, int(k))

    def _decide(self, lower_bounds_all, upper_bounds_all, dual_vars, primal_input, primals, layers, mask, k):
        mask = [(i == -1).float() for i in mask]                     # graph_score.py:22-24
        mask_1d = torch.cat([i for i in mask], 0).unsqueeze(0)
        start = time.time()
        dev = next(self.model.parameters()).device
        lower_bounds_all = [torch.as_tensor(i).to(dev) for i in lower_bounds_all]
        upper_bounds_all = [torch.as_tensor(i).to(dev) for i in upper_bounds_all]
        dual_vars = [torch.as_tensor(i).to(dev) for i in dual_vars]
        primal_input = torch.as_tensor(primal_input).to(dev)
        primals = [torch.as_tensor(i, dtype=torch.float32).to(dev) for i in primals]   # python-float lists, :30
        with torch.no_grad():
            fr = Frontier.from_reference_args(lower_bounds_all, upper_bounds_all, dual_vars, primals, primal_input,
                                              layers, mask_1d.to(dev))
            if k is None:
                _, idx, _ = self.model.score_frontier(fr, return_scores=False)
            else:
                _, idx, _ = self.model.score_frontier_topk(fr, k, return_scores=False)
        flat = [int(i) for i in idx.reshape(-1).tolist()]
        if self.verbose:
            print(f'graph requires: {time.time() - start}')
        if flat[0] < 0:   # the reference's torch.max raises on an empty candidate set (graph_score.py:41)
            raise RuntimeError('max(): no undecided ReLU (mask has no -1 entry)')
        return [flat_to_layer_index(f, self.hidden_sizes) for f in flat if f >= 0]
