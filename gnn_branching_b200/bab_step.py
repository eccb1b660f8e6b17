"""One batched branch-and-bound step, device-resident: pick -> split -> bound -> score -> add.

The reference's loop body (plnn/relu_conv_gnnkwthreshold.py:126-244) handles ONE domain per iteration: ``pick_out`` the domain
with the smallest lower bound, build its two children with ``net.get_lower_bound(mask, lbs, ubs, decision, choice)``
(= ``KWConvGen.update_the_model``: intermediate bounds, then a Gurobi LP), ask the GNN for each child's branching decision
(``graph.decision``) and ``add_domain`` the children that can still violate the property.  ``FrontierStep.step`` does the same
for the next ``max_B`` domains of the queue at once, and nothing but four integers crosses the PCIe bus:

    DomainQueue.pick(max_B)            gnnb_queue_pick       the parents' bounds, masks and stored decisions, dense [B, .]
    split on the stored decision       (index arithmetic)    2 B children: (parent, choice 0) and (parent, choice 1)
    Scorer.child_bounds                gnnb_child_bounds     bounds part of update_the_model for the 2 B children + BaB masks
    GraphNet.score_frontier            gnnb_score            each child's GNN decision (argmax over its undecided ReLUs)
    DomainQueue.add(children, keep)    gnnb_queue_add        children whose lower bound is still below the decision bound

With ``kw_fallback=True`` the step also carries the reference's threshold rule (:145-203): where the GNN's split improved the
lower bound by less than ``branching_threshold`` (``(min(lb0, 0) + min(lb1, 0) - 2 lb) / (-2 lb)``), the BaBSR / KW heuristic's
decision (``gnnb_babsr`` = ``choose_node_conv``) is tried on the same parent — unless that ReLU has already proved ineffective
``kwbd_threshold`` times — and replaces the GNN's when its children improve the bound more; a KW decision that does worse than
the GNN's and improves by less than 0.05 is counted as ineffective.  The counters live on the device, per ReLU (the reference
keeps a dict keyed by "layer-index"); the intercept counter of ``choose_node_conv`` (``icp_score``), which the reference carries
from one iteration to the next, starts at zero for every parent of a batch.

With ``strong_branching_k`` > 1 or ``strong_branching_kw_k`` > 0 the step does strong branching over a short candidate list
instead (the filtered strong branching of OVAL's later FSB rule; the GNN was trained to imitate strong branching): the parents
are scored again with ``gnnb_score_topk`` on the frontier their decision came from, the candidates are the GNN's ranks
0 .. k - 1 followed by the top ``strong_branching_kw_k`` ReLUs of the BaBSR score term (``gnnb_babsr``'s dense |score|, ranked
with ``gnnb_topk`` over the parent's undecided ReLUs) that are not in the list yet, and each parent keeps the split whose
children improve its lower bound most (the improvement formula of the threshold rule; ties keep the earlier rank).  Rank 0
is the stored decision, whose children the step bounds anyway; every further rank costs one ``gnnb_child_bounds`` call on the
parents that have such a candidate.  The improvement is measured on the KW / interval surrogate bounds of the children, not
on the LP bounds the reference would compute (see below).  Strong branching and the threshold rule are exclusive.

With ``online=True`` (which needs ``kw_fallback=True``: the threshold rule is the trigger) the step also fine-tunes the GNN
online, as the reference's ``--bab_online`` loop does (plnn/relu_conv_online.py:198-211 with GraphChoice.online_learning,
graphnet/graph_score_online.py:62-77): when the KW decision of m > 0 parents replaced their GNN decision, one Adam step
(``online_lr``, ``online_wd``: the reference's ``GraphChoice(lr=1e-4, wd=1e-4)``) is taken on the loss
``(1/m) sum_parents (gnn_score - kw_score)`` over the parents' GNN frontier, with the gradient pass of
``gnnb_score_grad_device`` on terms built on the device; the children are then decided by the updated GNN, as in the
reference, where ``online_learning`` precedes the children's ``decision`` calls.  The updated parameters are copied device to
device into ``model``, so ``state_dict()`` follows the fine-tuning.  Where this differs from the reference:
  - one Adam step on the mean loss of a batch, not one step per parent; the mean keeps the single-parent gradient scale, so
    the weight decay weighs as in the reference;
  - the + term is the parent's stored GNN decision.  The reference differentiates the scores of its last ``decision()`` call,
    a one-at-a-time detail with no batched counterpart;
  - the reference driver's constant ``pref_online_thd = 2`` (SURVEY §5) is not modelled: its use in relu_conv_online.py
    could not be checked against the reference source.

What is NOT here is the LP: Gurobi is out of scope (SURVEY §8), so the values the reference takes from the LP solution are
SURROGATES and the step is labelled as such wherever it is reported — the child's lower bound is the lower bound of the
property output from the KW / interval pass (valid, but looser than the LP's), its upper bound is the parent's, the GNN's
LP features are zero duals and the activations of the ball centre as primals (the convention of the synthetic frontier
generator, SURVEY §8d).  A branch-and-bound run built from these steps is therefore a sound but weaker verifier than the
reference's; its purpose here is the data path: the bounds the scorer reads are produced on the GPU that scores them.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List

import torch
import torch.nn.functional as F

from . import _lib
from .domain_queue import DomainBatch, DomainQueue
from .frontier import Frontier
from .graph_conv import GraphNet
from .networks import NetSpec


@dataclass
class StepStats:
    picked: int              # parents taken from the queue
    children: int            # 2 * picked
    second_pass: int         # children whose interval bounds triggered the second KW pass
    infeasible: int          # children dropped because their bounds cross (or pin a node to exactly zero)
    added: int               # children put back into the queue
    global_lb: float         # smallest lower bound left in the queue (nan when it is empty)
    kw_tried: int = 0        # parents whose GNN split improved too little: the KW decision was bounded as well
    kw_used: int = 0         # ... and won
    sb_bounded: int = 0      # strong branching: child pairs bounded beyond the stored decision's
    sb_changed: int = 0      # strong branching: parents whose split is not the stored GNN decision
    online_trained: int = 0  # online: parents whose loss terms went into this step's Adam step (= kw_used)


class FrontierStep:
    def __init__(self, model: GraphNet, net: NetSpec, x: torch.Tensor, eps: float, Wp: torch.Tensor, bp: float,
                 capacity: int = 1 << 16, decision_bound: float = 0.0, device: int = 0, kw_fallback: bool = False,
                 branching_threshold: float = 0.2, kwbd_threshold: int = 20, sparsest_layer: int = 0, strong_branching_k: int = 1,
                 strong_branching_kw_k: int = 0, online: bool = False, online_lr: float = 1e-4, online_wd: float = 1e-4):
        self.model, self.net, self.eps, self.decision_bound = model, net, float(eps), float(decision_bound)
        self.kw_fallback, self.branching_threshold, self.kwbd_threshold = bool(kw_fallback), float(branching_threshold), int(kwbd_threshold)
        self.sparsest_layer = int(sparsest_layer)
        self.sb_k, self.sb_kw_k = int(strong_branching_k), int(strong_branching_kw_k)
        if not 1 <= self.sb_k <= _lib.TOPK_MAX or not 0 <= self.sb_kw_k <= _lib.TOPK_MAX:
            raise ValueError(f'strong_branching_k must be in [1, {_lib.TOPK_MAX}] and strong_branching_kw_k in [0, {_lib.TOPK_MAX}]')
        self.strong = self.sb_k > 1 or self.sb_kw_k > 0
        if self.strong and self.kw_fallback:
            raise ValueError('strong branching and kw_fallback (the threshold rule) cannot be combined')
        self.last_strong = None          # (candidates [B, K, 2], improvement [B, K], chosen rank [B]) of the last strong step
        self.online, self.online_lr, self.online_wd = bool(online), float(online_lr), float(online_wd)
        if self.online and not self.kw_fallback:
            raise ValueError('online=True needs kw_fallback=True: the threshold rule triggers the online update')
        # (parent rows in the step's pick order, GNN flat index, KW flat index, term scores [2 m]) of the last online update
        self.last_online = None
        self.dev = torch.device('cuda', device)
        self.scorer = model.scorer(device)
        self.scorer.set_network(net, key=net.key)
        self.queue = DomainQueue(self.scorer, capacity)
        self.x = x.reshape(1, -1).to(self.dev, torch.float32)
        self.Wp = Wp.reshape(1, -1).to(self.dev, torch.float32)
        self.bp = torch.tensor([float(bp)], device=self.dev)
        self.sizes = [net.n0] + net.hidden_sizes + [1]
        self.offsets = torch.tensor([0] + list(torch.tensor(net.hidden_sizes).cumsum(0)), device=self.dev)
        # surrogate LP primals: the activations of the ball centre (pre- and post-ReLU), shared by every domain
        pre, post, h = [], [], self.x.reshape(1, *net.input_shape)
        for a in net.affine:
            w, b = a.weight.to(self.dev), a.bias.to(self.dev)
            h = F.conv2d(h, w, b, stride=a.stride, padding=a.padding) if a.kind == 'conv' else F.linear(h.reshape(1, -1), w, b)
            pre.append(h.reshape(1, -1))
            h = h.clamp(min=0)
            post.append(h.reshape(1, -1))
        self.prim_pre, self.prim_post = pre, post
        self.prim_out = (post[-1] @ self.Wp.t()).reshape(1) + self.bp
        self._zeros = {}
        self.ineff_kw = torch.zeros(net.n_hidden, dtype=torch.int32, device=self.dev)      # relu_conv_gnnkwthreshold.py:134 ineff_kw_dc
        if self.online:
            self.scorer.adam_reset()     # a fresh optimiser per run, as the reference builds GraphChoice per verification

    # ---- seeding ----
    def seed_root(self, lbs: List[torch.Tensor] = None, ubs: List[torch.Tensor] = None) -> None:
        """Put the root domain into the queue: its bounds (L + 2 flat tensors; computed on the device by ``gnnb_root_bounds``, the
        bounds part of ``build_the_model``, when not given), mask from the bounds, GNN decision."""
        if lbs is None:
            lbs, ubs, _, _ = self.scorer.root_bounds(self.x, self.eps, self.Wp, self.bp, with_mask=False)
        lb = [t.reshape(1, -1).to(self.dev, torch.float32) for t in lbs]
        ub = [t.reshape(1, -1).to(self.dev, torch.float32) for t in ubs]
        mask = torch.cat([self._bab_mask(lb[k], ub[k]) for k in range(1, self.net.L + 1)], dim=1)
        dec, ok = self._decide(lb, ub, mask)
        self.queue.add(DomainBatch(lb[-1].reshape(1).clone(), ub[-1].reshape(1).clone(), lb, ub, mask, dec), keep=ok)

    # ---- the step ----
    def step(self, max_B: int, threshold: float = float('inf')) -> StepStats:
        L = self.net.L
        parents = self.queue.pick(max_B, threshold)
        B = parents.B
        if B == 0:
            return StepStats(0, 0, 0, 0, 0, float('nan'))
        rep = lambda t: t.repeat_interleave(2, dim=0)
        choice = torch.arange(2 * B, device=self.dev, dtype=torch.int32) & 1
        dec = rep(parents.decision)
        lbs, ubs, masks, second = self.scorer.child_bounds(self.x, self.eps, self.Wp.expand(2 * B, -1), self.bp.expand(2 * B),
                                                           [rep(t) for t in parents.lb], [rep(t) for t in parents.ub],
                                                           dec[:, 0], dec[:, 1], choice)
        kw_tried = kw_used = sb_bounded = sb_changed = 0
        self.last_online = None
        if self.kw_fallback:
            kw_tried, kw_used = self._kw_fallback(parents, lbs, ubs, masks, second)
        elif self.strong:
            sb_bounded, sb_changed = self._strong_branching(parents, lbs, ubs, masks, second)
        # ReLUs the ancestors fixed stay fixed (their bounds say so already); this child's own split is in `masks` too, because
        # its bound is exactly 0 on the fixed side (conv_kwinter_gen.py:572: relu_mask[decision] = choice)
        mask = torch.cat(masks, dim=1)
        # Infeasible children (the split contradicts the parent's other constraints: intersected bounds cross, l > u) are where the
        # reference's LP reports infeasibility and the child is never added; here they are dropped by the same sign.  So are
        # children with a node pinned to exactly zero from both sides (l = u = 0): compute_ratio is 0 / 0 there, in the
        # reference as well (its NaN trap, graph_conv.py:184-186).  Neither kind may reach the scorer, whose NaN flag is an error:
        # they are scored on their parent's bounds instead (no host round trip to compact them away) and then not kept.
        bad = lbs[L + 1].reshape(-1) > ubs[L + 1].reshape(-1)
        for k in range(1, L + 1):
            bad |= ((lbs[k] > ubs[k]) | ((lbs[k] >= 0) & (ubs[k] <= 0))).any(dim=1)
        sel = bad[:, None]
        s_lbs = [torch.where(sel, rep(p), c) for p, c in zip(parents.lb, lbs)]
        s_ubs = [torch.where(sel, rep(p), c) for p, c in zip(parents.ub, ubs)]
        new_dec, ok = self._decide(s_lbs, s_ubs, torch.where(sel, rep(parents.mask), mask))
        lower = lbs[L + 1].reshape(-1)
        keep = ok & ~bad & (lower < self.decision_bound)
        children = DomainBatch(lower.contiguous(), rep(parents.upper_bound).contiguous(), lbs, ubs, mask, new_dec)
        added = self.queue.add(children, keep=keep)
        glb = self.queue.global_lb if len(self.queue) else float('nan')
        return StepStats(B, 2 * B, int(second.sum()), int(bad.sum()), added, glb, kw_tried, kw_used, sb_bounded, sb_changed,
                         kw_used if self.online else 0)

    # ---- the threshold rule (relu_conv_gnnkwthreshold.py:145-203) ----
    def _improvement(self, plb: torch.Tensor, lbs, ubs) -> torch.Tensor:
        """(min(lb0, 0) + min(lb1, 0) - 2 lb) / (-2 lb) per parent from its two children's output bounds; an infeasible child
        (crossing output bounds) counts as fully resolved (min(., 0) = 0); parents with lb >= 0 need no fallback (1)."""
        L = self.net.L
        low = lbs[L + 1].reshape(-1)
        low = torch.where(low > ubs[L + 1].reshape(-1), torch.zeros_like(low), low).clamp(max=0)
        imp = (low[0::2] + low[1::2] - 2 * plb) / (-2 * plb)
        return torch.where(plb < 0, imp, torch.ones_like(imp))

    def _kw_fallback(self, parents: DomainBatch, lbs, ubs, masks, second):
        """Replaces, in place, the children of the parents whose KW decision beats their GNN decision.  One count is read back
        (how many parents need the second opinion)."""
        from .kw_score_conv import babsr_frontier
        L, dev = self.net.L, self.dev
        gnn_imp = self._improvement(parents.lower_bound, lbs, ubs)
        idx = (gnn_imp < self.branching_threshold).nonzero().view(-1)
        m = int(idx.numel())
        if m == 0:
            return 0, 0
        plb_all = [t[idx] for t in parents.lb]
        pub_all = [t[idx] for t in parents.ub]
        pmask = parents.mask[idx]
        empty = torch.empty(0, device=dev)
        fr = Frontier(net=self.net, lb=plb_all, ub=pub_all, dual=[], prim_pre=[], prim_post=[], prim_out=empty, primal_input=empty,
                      Wp=self.Wp.expand(m, -1).contiguous(), bp=self.bp.expand(m).contiguous(), mask=(pmask == -1).float())
        kw_dec, _, _, _ = babsr_frontier(fr, None, None, self.sparsest_layer, scorer=self.scorer)
        flat = (self.offsets[kw_dec[:, 0].clamp(min=0).long()] + kw_dec[:, 1].clamp(min=0).long())
        gnn_dec = parents.decision[idx]
        ok = (kw_dec[:, 0] >= 0) & (self.ineff_kw[flat] < self.kwbd_threshold) & (kw_dec != gnn_dec).any(dim=1)
        # parents without a usable KW decision are bounded on their GNN decision again (no second count read back); their result
        # is discarded
        kw_imp, use = self._try_split(parents.lower_bound[idx], plb_all, pub_all, idx, torch.where(ok[:, None], kw_dec, gnn_dec),
                                      gnn_imp[idx], ok, lbs, ubs, masks, second)                  # :177-190
        bad_kw = ok & (kw_imp < gnn_imp[idx]) & (kw_imp < 0.05)                                   # :171-176
        self.ineff_kw.index_add_(0, flat, bad_kw.to(torch.int32))
        used = int(use.sum())
        if self.online and used:
            self._online_update(parents, idx, use, self.offsets[gnn_dec[:, 0].long()] + gnn_dec[:, 1].long(), flat, used)
        return m, used

    def _online_update(self, parents: DomainBatch, idx, use, gnn_flat, kw_flat, used: int):
        """One Adam step on (1/m) sum (score at the stored GNN decision - score at the KW decision) over the ``used`` parents
        (rows ``idx[use]``) on the parents' GNN frontier (graph_score_online.py:62-77), then the new parameters into
        ``model``.  The 2 len(idx) terms are built on the device; parents where KW did not win get inactive terms (domain -1)."""
        dom = torch.where(use, idx, torch.full_like(idx, -1)).to(torch.int32)
        coeff = torch.full((idx.numel(),), 1.0 / used, dtype=torch.float32, device=self.dev)
        terms = (torch.cat([dom, dom]), torch.cat([gnn_flat, kw_flat]).to(torch.int32), torch.cat([coeff, -coeff]))
        fr = self._frontier(parents.lb, parents.ub, parents.mask)
        vals = self.scorer.score_grad(fr, terms)
        self.scorer.adam_step(self.online_lr, weight_decay=self.online_wd)
        self.model.adopt_weights(self.scorer)
        n = idx.numel()
        self.last_online = (idx[use], gnn_flat[use], kw_flat[use], torch.cat([vals[:n][use], vals[n:][use]]))

    def _try_split(self, plower, plb, pub, idx, dec, beat, ok, lbs, ubs, masks, second):
        """Bound the two children of the parents ``idx`` (lower bounds ``plower``, bounds ``plb`` / ``pub``: [m, .]) split on
        ``dec`` ([m, 2] (layer, index)) and, in place, replace the current children (rows 2 idx, 2 idx + 1 of lbs / ubs / masks /
        second) of those where ``ok`` holds and the new split improves the bound strictly more than ``beat`` [m].  Returns the new
        split's improvement [m] and where it replaced the children [m]."""
        L, dev, m = self.net.L, self.dev, int(idx.numel())
        rep = lambda t: t.repeat_interleave(2, dim=0)
        choice = torch.arange(2 * m, device=dev, dtype=torch.int32) & 1
        d = rep(dec)
        k_lbs, k_ubs, k_masks, k_second = self.scorer.child_bounds(self.x, self.eps, self.Wp.expand(2 * m, -1), self.bp.expand(2 * m),
                                                                   [rep(t) for t in plb], [rep(t) for t in pub],
                                                                   d[:, 0], d[:, 1], choice)
        imp = self._improvement(plower, k_lbs, k_ubs)
        use = ok & (imp > beat)
        rows = rep(2 * idx) + (torch.arange(2 * m, device=dev) & 1)
        sel = rep(use)
        for k in range(1, L + 2):
            lbs[k][rows] = torch.where(sel[:, None], k_lbs[k], lbs[k][rows])
            ubs[k][rows] = torch.where(sel[:, None], k_ubs[k], ubs[k][rows])
        for k in range(L):
            masks[k][rows] = torch.where(sel[:, None], k_masks[k], masks[k][rows])
        second[rows] = torch.where(sel, k_second, second[rows])
        return imp, use

    # ---- strong branching over the GNN's (and BaBSR's) top candidates ----
    def _strong_branching(self, parents: DomainBatch, lbs, ubs, masks, second):
        """Replaces, in place, the children of every parent by those of its best candidate split (largest improvement, earliest
        rank on ties).  One count is read back per rank beyond 0.  Returns (child pairs bounded, parents whose split changed)."""
        from .kw_score_conv import babsr_frontier
        B, dev = parents.B, self.dev
        fr = self._frontier(parents.lb, parents.ub, parents.mask)
        _, cand, _ = self.model.score_frontier_topk(fr, self.sb_k, return_scores=False)
        if self.sb_kw_k:
            _, _, _, kw_scores = babsr_frontier(fr, None, None, self.sparsest_layer, return_scores=True, scorer=self.scorer)
            _, kw_cand = self.scorer.topk(kw_scores, self.sb_kw_k, mask=fr.mask)
            cand = torch.cat([cand, kw_cand], dim=1)
        K = int(cand.shape[1])
        # the list: GNN ranks first, then the BaBSR candidates not in it yet; empty slots and repeats are skipped (-1)
        cand = cand.long()
        for r in range(self.sb_k, K):
            dup = ((cand[:, :r] == cand[:, r:r + 1]) & (cand[:, r:r + 1] >= 0)).any(dim=1)
            cand[:, r] = torch.where(dup, torch.full_like(cand[:, r], -1), cand[:, r])
        lay = torch.bucketize(cand.clamp(min=0), self.offsets[1:], right=True)
        dec = torch.stack([lay, cand.clamp(min=0) - self.offsets[lay]], dim=2).to(torch.int32)
        dec = torch.where((cand >= 0)[:, :, None], dec, torch.full_like(dec, -1))
        imp = torch.full((B, K), float('-inf'), device=dev)
        imp[:, 0] = self._improvement(parents.lower_bound, lbs, ubs)           # rank 0: the stored decision's children
        best = imp[:, 0].clone()
        chosen = torch.zeros(B, dtype=torch.long, device=dev)
        bounded = 0
        for r in range(1, K):
            idx = (cand[:, r] >= 0).nonzero().view(-1)
            m = int(idx.numel())
            if m == 0:
                continue
            bounded += m
            r_imp, use = self._try_split(parents.lower_bound[idx], [t[idx] for t in parents.lb], [t[idx] for t in parents.ub], idx,
                                         dec[idx, r], best[idx], torch.ones(m, dtype=torch.bool, device=dev), lbs, ubs, masks, second)
            imp[idx, r] = r_imp
            best[idx] = torch.where(use, r_imp, best[idx])
            chosen[idx] = torch.where(use, torch.full_like(chosen[idx], r), chosen[idx])
        self.last_strong = (dec, imp, chosen)
        split = dec[torch.arange(B, device=dev), chosen]
        changed = int(((chosen > 0) & (split != parents.decision).any(dim=1)).sum())
        return bounded, changed

    # ---- helpers ----
    @staticmethod
    def _bab_mask(l: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
        """conv_kwinter_gen.py:696-713: passing 1, blocked 0, ambiguous -1."""
        one, zero = torch.ones_like(l, dtype=torch.int8), torch.zeros_like(l, dtype=torch.int8)
        return torch.where((l >= 0) & (u >= 0), one, torch.where((l <= 0) & (u <= 0), zero, -one))

    def _frontier(self, lbs, ubs, mask) -> Frontier:
        """The GNN's frontier of n domains: their bounds, the BaB mask's undecided ReLUs as candidates, and the surrogate LP
        features (zero duals, the ball centre's activations as primals)."""
        n = int(mask.shape[0])
        L = self.net.L
        z = self._zeros.get(n)
        if z is None:
            z = [torch.zeros(n, s, 3, device=self.dev) for s in self.sizes[1:L + 1]]
            self._zeros = {n: z}
        ex = lambda t: t.expand(n, -1).contiguous()
        return Frontier(net=self.net, lb=lbs, ub=ubs, dual=z, prim_pre=[ex(t) for t in self.prim_pre], prim_post=[ex(t) for t in self.prim_post],
                        prim_out=self.prim_out.expand(n).contiguous(), primal_input=ex(self.x), Wp=ex(self.Wp), bp=self.bp.expand(n).contiguous(),
                        mask=(mask == -1).float())

    def _decide(self, lbs, ubs, mask):
        """GNN decision of every domain (graph_score.py:21-56 batched): [n, 2] int32 (layer, index), and which domains have
        an undecided ReLU at all."""
        fr = self._frontier(lbs, ubs, mask)
        _, idx, _ = self.model.score_frontier(fr, return_scores=False)
        ok = idx >= 0
        flat = idx.clamp(min=0).long()
        lay = torch.bucketize(flat, self.offsets[1:], right=True)
        dec = torch.stack([lay, flat - self.offsets[lay]], dim=1).to(torch.int32)
        return dec, ok
