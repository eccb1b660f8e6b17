"""Top-k branching candidates (gnnb_topk, gnnb_score_topk, Scorer.score_topk / topk, GraphChoice.decision_topk) and strong
branching in FrontierStep.

The order contract, written out in `_ref_order`: the candidates of a row are its entries with mask != 0 (a -inf score is still a
candidate); NaN scores come first in ascending index, then the other candidates by score, descending, equal scores (-0.0 ==
+0.0) by ascending index; a returned score is the bit pattern of the score at the returned index; slots past the last candidate
hold (-inf, -1).  Entry 0 is gnnb_score's (best_score, best_idx) bit for bit.
"""
import ctypes as C
import functools
import os

import numpy as np
import pytest
import torch

from golden_io import ARCHS, GOLDEN, load_gnn, load_root
from gnn_branching_b200 import GraphNet, GraphChoice, Scorer, synthetic_frontier, _lib
from oracle import graphnet_oracle as O

pytestmark = pytest.mark.gpu

KS = [1, 2, 5, 16, 63, 64]


def _bits(t):
    return t.contiguous().view(torch.int32)


def _ref_order(scores, mask):
    """Candidate indices of every row in contract order, padded with -1: [B, n] int64 (torch reference, float64 on the GPU)."""
    B, n = scores.shape
    cand = torch.ones_like(scores, dtype=torch.bool) if mask is None else (mask != 0)
    nan = torch.isnan(scores)
    val = scores.double()
    val = torch.where(val == 0, torch.zeros_like(val), val)                   # -0.0 ties with +0.0
    val = torch.where(nan, torch.full_like(val, float('inf')), val)
    tier = torch.where(cand & nan, 2, torch.where(cand, 1, 0))                # NaN candidates, other candidates, the rest
    # stable sorts: by value descending, then by tier descending; equal (tier, value) keep ascending index
    order = torch.sort(val, dim=1, descending=True, stable=True).indices
    order = order.gather(1, torch.sort(tier.gather(1, order), dim=1, descending=True, stable=True).indices)
    return torch.where(tier.gather(1, order) > 0, order, torch.full_like(order, -1))


def _ref_topk(scores, mask, k, order=None):
    order = _ref_order(scores, mask) if order is None else order
    B, n = scores.shape
    idx = order[:, :k]
    if idx.shape[1] < k:
        idx = torch.cat([idx, torch.full((B, k - idx.shape[1]), -1, dtype=idx.dtype, device=idx.device)], dim=1)
    sc = torch.where(idx >= 0, scores.gather(1, idx.clamp(min=0)), torch.full(idx.shape, float('-inf'), device=scores.device))
    return sc, idx.to(torch.int32)


def _crafted(B, n, seed):
    """Rows with many exact ties, -0.0 / +0.0, NaN, +-inf and -inf candidates, all-masked rows and rows with fewer candidates
    than k.  Returns CUDA (scores, mask)."""
    g = torch.Generator().manual_seed(seed)
    gd = torch.Generator(device='cuda').manual_seed(seed)
    s = torch.randint(-4, 5, (B, n), generator=gd, device='cuda').float() * 0.25     # 9 distinct values: exact ties everywhere
    u = torch.rand(B, n, generator=gd, device='cuda')
    s = torch.where(u < 0.05, torch.full_like(s, -0.0), s)
    s = torch.where((u >= 0.05) & (u < 0.08), torch.full_like(s, float('nan')), s)
    s = torch.where((u >= 0.08) & (u < 0.10), torch.full_like(s, float('inf')), s)
    s = torch.where((u >= 0.10) & (u < 0.12), torch.full_like(s, float('-inf')), s)
    s = torch.where((u >= 0.12) & (u < 0.30), torch.randn(B, n, generator=gd, device='cuda'), s)
    mask = (torch.rand(B, n, generator=gd, device='cuda') < 0.6).float()
    rows = torch.randperm(B, generator=g)
    for j, b in enumerate(rows[:min(B, 8)].tolist()):
        kind = j % 4
        if kind == 0:
            mask[b] = 0                                                         # no candidate
        elif kind == 1:
            mask[b] = 0
            mask[b, torch.randperm(n, generator=g)[:3]] = 1                     # three candidates
        elif kind == 2:
            mask[b] = 0
            mask[b, 0] = 1
            s[b, 0] = float('-inf')                                             # only a -inf candidate
        else:
            s[b] = torch.where(torch.rand(n, generator=g) < 0.5, -0.0, 0.0).cuda()     # signed zeros only
    if B == 1 and n > 1:
        s[0, n // 2] = float('nan')
    return s, mask


@functools.lru_cache(maxsize=None)
def _bare_scorer():
    return Scorer(0)


@pytest.mark.parametrize('B,n', [(1, 1), (3000, 1), (1, 31), (3000, 31), (1, 3172), (3000, 3172), (1, 6756), (3000, 6756),
                                 (1, 100000), (3000, 100000)])
def test_topk_matches_reference(B, n):
    sc = _bare_scorer()
    scores, mask = _crafted(B, n, seed=B * 7 + n)
    for m in (mask, None):
        order = _ref_order(scores, m)
        for k in KS:
            got_s, got_i = sc.topk(scores, k, mask=m)
            want_s, want_i = _ref_topk(scores, m, k, order)
            assert torch.equal(got_i, want_i), (B, n, k, m is None)
            assert torch.equal(_bits(got_s), _bits(want_s)), (B, n, k, m is None)


def test_topk_crafted_rows_explicitly():
    """A few rows spelled out: ties, signed zeros, NaN first, -inf candidates, fewer than k candidates, none."""
    inf, nan = float('inf'), float('nan')
    s = torch.tensor([[1.0, 2.0, 2.0, 1.0, 2.0, 0.5],
                      [0.0, -0.0, 0.0, -0.0, -1.0, 1.0],
                      [-inf, 3.0, nan, inf, nan, -inf],
                      [5.0, 4.0, 3.0, 2.0, 1.0, 0.0],
                      [5.0, 4.0, 3.0, 2.0, 1.0, 0.0]], device='cuda')
    m = torch.tensor([[1, 1, 1, 1, 1, 1], [1, 1, 1, 1, 1, 1], [1, 1, 1, 1, 1, 1], [0, 1, 0, 0, 1, 0], [0, 0, 0, 0, 0, 0]],
                     dtype=torch.float32, device='cuda')
    ts, ti = _bare_scorer().topk(s, 5, mask=m)
    assert ti.tolist() == [[1, 2, 4, 0, 3], [5, 0, 1, 2, 3], [2, 4, 3, 1, 0], [1, 4, -1, -1, -1], [-1] * 5]
    assert _bits(ts[1, 1:]).tolist() == _bits(torch.tensor([0.0, -0.0, 0.0, -0.0])).tolist()
    assert torch.isnan(ts[2, :2]).all() and ts[2, 2] == inf and ts[2, 4] == -inf
    assert ts[3, 2:].eq(-inf).all() and ts[4].eq(-inf).all()


def _frontier(arch, B, seed, device='cuda'):
    net, lbs, ubs, wp, bp = load_root(arch)
    return synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=seed, device=device)


def _scorer(net, math='tc', fuse=1, chunk=0, rescore=False, weights='random'):
    sc = Scorer(0, math=math, chunk=chunk, rescore=rescore)
    sc.set_gnn(load_gnn(weights))
    sc.set_network(net, key=net.key)
    if math == 'tc':
        sc.set_option('fuse', fuse)
    return sc


@pytest.mark.parametrize('arch', ARCHS)
def test_k1_equals_argmax(arch):
    fr = _frontier(arch, 256, seed=11 + ARCHS.index(arch))
    fr.mask[3].zero_()                                       # one subdomain without a candidate
    sc = _scorer(fr.net)
    best, idx, scores = sc.score(fr)
    ts, ti = sc.topk(scores, 1, mask=fr.mask)
    assert torch.equal(ti[:, 0], idx) and torch.equal(_bits(ts[:, 0]), _bits(best))
    assert int(idx[3]) == -1


@pytest.mark.parametrize('chunk', [0, 16])
@pytest.mark.parametrize('mem', ['device', 'host'])
@pytest.mark.parametrize('fuse', [1, 0])
@pytest.mark.parametrize('math', ['tc', 'simt'])
@pytest.mark.parametrize('arch', ARCHS)
def test_score_topk_on_the_scoring_path(arch, math, fuse, mem, chunk):
    """B = 1 000: the last wave is ragged (chunk 16) and host buffers run the growing wave ramp."""
    fr = _frontier(arch, 1000, seed=300 + ARCHS.index(arch), device='cpu')
    fr.mask[7].zero_()
    fr.mask[8].zero_()
    fr.mask[8, 5] = 1                                        # a single candidate
    fr = fr.to('cuda') if mem == 'device' else fr.pin()
    sc = _scorer(fr.net, math=math, fuse=fuse, chunk=chunk)
    sc.score(fr)                                             # warm-up: workspace and result buffers
    n0 = sc.launches
    best, idx, dense = sc.score(fr)
    d_score = sc.launches - n0
    for k in (1, 5, 64):
        n0 = sc.launches
        ts, ti, s = sc.score_topk(fr, k, return_scores=True)
        assert sc.launches - n0 == d_score
        assert ts.shape == (fr.B, k) and ts.is_cuda == (mem == 'device')
        assert torch.equal(s, dense)
        assert torch.equal(ti[:, 0], idx) and torch.equal(_bits(ts[:, 0]), _bits(best))
        ws, wi = sc.topk(dense.cuda(), k, mask=fr.mask.cuda())
        assert torch.equal(ti.cuda(), wi) and torch.equal(_bits(ts.cuda()), _bits(ws))
        assert int(ti[7, 0]) == -1 and int(ti[8, 0]) == 5 and (k == 1 or int(ti[8, 1]) == -1)
    ts2, ti2, none = sc.score_topk(fr, 5)                    # without dense scores
    assert none is None and torch.equal(ti2, sc.score_topk(fr, 5)[1])


def test_score_topk_against_oracle():
    """The top-k index set agrees with the oracle's wherever the oracle's gap between rank k and rank k + 1 exceeds
    1e-4 * max|s|."""
    sd = load_gnn('random')
    for arch in ARCHS:
        fr = _frontier(arch, 24, seed=77 + ARCHS.index(arch), device='cpu')
        s_or, _ = O.gnn_forward(sd, fr)
        sc = _scorer(fr.net)
        for k in (4, 16):
            _, ti, _ = sc.score_topk(fr.to('cuda'), k)
            ti = ti.cpu()
            checked = 0
            for b in range(fr.B):
                cand = fr.mask[b].nonzero().view(-1)
                v = s_or[b][cand].double()
                order = torch.argsort(v, descending=True)
                scale = float(v.abs().max())
                if cand.numel() > k and float(v[order[k - 1]] - v[order[k]]) <= 1e-4 * scale:
                    continue
                want = set(cand[order[:k]].tolist())
                assert set(x for x in ti[b].tolist() if x >= 0) == want, (arch, k, b)
                checked += 1
            assert checked >= fr.B // 2, (arch, k, checked)


ROWS = [2, 17, 40, 63]


@functools.lru_cache(maxsize=None)
def _overflow_case():
    """The overflow construction of option "rescore": a seeded base x 64 frontier whose subdomains ROWS have their duals scaled
    by the smallest power of ten at which the tensor-core pass reports NaN while the fp32 SIMT mode stays finite."""
    net = load_root('base')[0]
    tc, simt = _scorer(net), _scorer(net, math='simt')
    for f in (1e6, 1e7, 1e8, 1e9, 1e10):
        fr = _frontier('base', 64, seed=4000, device='cpu')
        for d in fr.dual:
            d[torch.tensor(ROWS)] *= f
        tc.score(fr.to('cuda'), return_scores=False, check=False)
        n = C.c_int64(0)
        st = tc.lib.gnnb_check(tc.h, C.c_void_p(torch.cuda.current_stream().cuda_stream), C.byref(n))
        if st != _lib.GNNB_ERR_NAN:
            continue
        _, _, s = simt.score(fr.to('cuda'))
        if bool(torch.isfinite(s[ROWS]).all()):
            return fr
    pytest.fail('no factor overflows the tensor-core path with a finite fp32 result')


@pytest.mark.parametrize('chunk', [0, 16])
@pytest.mark.parametrize('mem', ['device', 'host'])
def test_rescore_gives_fp32_topk(mem, chunk):
    fr = _overflow_case()
    k = 8
    ref_tc = _scorer(fr.net).score_topk(fr.to('cuda'), k, check=False)
    torch.cuda.synchronize()
    ref_simt = _scorer(fr.net, math='simt').score_topk(fr.to('cuda'), k)
    sc = _scorer(fr.net, chunk=chunk, rescore=True)
    ts, ti, s = sc.score_topk(fr.to('cuda') if mem == 'device' else fr.pin(), k, return_scores=True)
    assert sc.rescored == len(ROWS)
    ts, ti = ts.cuda(), ti.cuda()
    keep = torch.ones(fr.B, dtype=torch.bool, device='cuda')
    keep[ROWS] = False
    assert torch.equal(ti[ROWS], ref_simt[1][ROWS]) and torch.equal(_bits(ts[ROWS]), _bits(ref_simt[0][ROWS]))
    assert torch.equal(ti[keep], ref_tc[1][keep]) and torch.equal(_bits(ts[keep]), _bits(ref_tc[0][keep]))
    ws, wi = sc.topk(s.cuda(), k, mask=fr.mask.cuda())
    assert torch.equal(wi, ti) and torch.equal(_bits(ws), _bits(ts))


def test_invalid_arguments():
    fr = _frontier('base', 4, seed=1)
    sc = _scorer(fr.net)
    d, keep = sc._frontier_desc(fr)
    out_s = torch.empty(4, 64, device='cuda')
    out_i = torch.empty(4, 64, dtype=torch.int32, device='cuda')
    scores = torch.randn(4, 10, device='cuda')
    fp, ip = _lib.fptr, (lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_int32)))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n0 = sc.launches
    for k in (0, 65, -1):
        assert sc.lib.gnnb_score_topk(sc.h, C.byref(d), k, fp(out_s), ip(out_i), None, st) == _lib.GNNB_ERR_INVALID
        assert sc.lib.gnnb_topk(sc.h, 4, 10, fp(scores), None, k, fp(out_s), ip(out_i), st) == _lib.GNNB_ERR_INVALID
    assert sc.lib.gnnb_score_topk(sc.h, C.byref(d), 4, None, ip(out_i), None, st) == _lib.GNNB_ERR_INVALID
    assert sc.lib.gnnb_score_topk(sc.h, C.byref(d), 4, fp(out_s), None, None, st) == _lib.GNNB_ERR_INVALID
    assert sc.lib.gnnb_topk(sc.h, 4, 10, fp(scores), None, 4, None, ip(out_i), st) == _lib.GNNB_ERR_INVALID
    assert sc.lib.gnnb_topk(sc.h, 4, 10, fp(scores), None, 4, fp(out_s), None, st) == _lib.GNNB_ERR_INVALID
    assert sc.lib.gnnb_topk(sc.h, 4, 10, None, None, 4, fp(out_s), ip(out_i), st) == _lib.GNNB_ERR_INVALID
    assert sc.lib.gnnb_topk(sc.h, -1, 10, fp(scores), None, 4, fp(out_s), ip(out_i), st) == _lib.GNNB_ERR_INVALID
    assert sc.lib.gnnb_topk(sc.h, 4, -1, fp(scores), None, 4, fp(out_s), ip(out_i), st) == _lib.GNNB_ERR_INVALID
    d.B = -1
    assert sc.lib.gnnb_score_topk(sc.h, C.byref(d), 4, fp(out_s), ip(out_i), None, st) == _lib.GNNB_ERR_INVALID
    d.B = 0
    assert sc.lib.gnnb_score_topk(sc.h, C.byref(d), 4, fp(out_s), ip(out_i), None, st) == _lib.GNNB_OK
    assert sc.lib.gnnb_topk(sc.h, 0, 10, fp(scores), None, 4, fp(out_s), ip(out_i), st) == _lib.GNNB_OK
    assert sc.launches == n0
    with pytest.raises(ValueError):
        sc.score_topk(fr, 65)
    with pytest.raises(ValueError):
        sc.topk(scores, 0)
    del keep


def test_null_frontier_arrays_are_rejected():
    """A frontier with one null array (a bound, a dual, the input point, the mask) fails gnnb_score, gnnb_score_winners and
    gnnb_score_topk with GNNB_ERR_INVALID before anything is enqueued, with DEVICE and HOST descriptors, and the context
    scores a valid frontier afterwards.  gnnb_score_grad rejects a null bound but does not read the mask."""
    fr = _frontier('base', 4, seed=2, device='cpu')
    sc = _scorer(fr.net)
    fp, ip = _lib.fptr, (lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_int32)))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    winners = torch.empty(4, 2, dtype=torch.int32, device='cuda')

    def desc_without(f, field, k=None):
        d, keep = sc._frontier_desc(f)
        if k is None:
            setattr(d, field, None)
        else:
            getattr(d, field)[k] = None                          # the per-layer table lives in `keep`
        return d, keep

    for mem, f in (('device', fr.to('cuda')), ('host', fr.pin())):
        want_best, want_idx, _ = sc.score(f, return_scores=False)
        best = torch.empty(4, 64, device=f.device, pin_memory=mem == 'host')
        idx = torch.empty(4, 64, dtype=torch.int32, device=f.device, pin_memory=mem == 'host')
        for name in (('lb', 1), ('dual', 2), ('primal_input',), ('mask',)):
            d, keep = desc_without(f, *name)
            n0 = sc.launches
            assert sc.lib.gnnb_score(sc.h, C.byref(d), fp(best), ip(idx), None, st) == _lib.GNNB_ERR_INVALID, (mem, name)
            assert sc.lib.gnnb_score_winners(sc.h, C.byref(d), C.c_void_p(winners.data_ptr()), None, st) == _lib.GNNB_ERR_INVALID
            assert sc.lib.gnnb_score_topk(sc.h, C.byref(d), 5, fp(best), ip(idx), None, st) == _lib.GNNB_ERR_INVALID
            assert sc.launches == n0, (mem, name)
            d.B = 0                                              # an empty frontier is never read
            assert sc.lib.gnnb_score(sc.h, C.byref(d), fp(best), ip(idx), None, st) == _lib.GNNB_OK
            del keep
            got_best, got_idx, _ = sc.score(f, return_scores=False)
            assert torch.equal(got_idx, want_idx) and torch.equal(_bits(got_best), _bits(want_best)), (mem, name)
        term = ((C.c_int32 * 1)(1), (C.c_int32 * 1)(5), (C.c_float * 1)(1.0), (C.c_float * 1)())
        for name, status in ((('lb', 1), _lib.GNNB_ERR_INVALID), (('mask',), _lib.GNNB_OK)):
            d, keep = desc_without(f, *name)
            n0 = sc.launches
            assert sc.lib.gnnb_score_grad(sc.h, C.byref(d), 1, *term, st) == status, (mem, name)
            assert (sc.launches == n0) == (status != _lib.GNNB_OK), (mem, name)
            del keep


def test_decision_topk(tmp_path):
    fr = _frontier('base', 3, seed=21, device='cpu')
    fr.mask[2].zero_()
    fr.mask[2, torch.tensor([4, 3000, 3100])] = 1              # three candidates, in the second and third layers
    ckpt = os.path.join(tmp_path, 'gnn.pt')
    torch.save(load_gnn('shipped'), ckpt)
    for b in range(fr.B):
        lbs, ubs, duals, primals, pin, layers, masks = fr.slice(b, b + 1).to_reference_args()
        init_mask, off = [], 0
        for n in fr.net.hidden_sizes:
            m = masks[0, off:off + n]
            init_mask.append(torch.where(m != 0, torch.full_like(m, -1), torch.ones_like(m)).int())
            off += n
        gc = GraphChoice(init_mask, ckpt)
        dec = gc.decision(lbs, ubs, duals, pin, [q.tolist() for q in primals], layers, init_mask)
        n_cand = int(fr.mask[b].sum())
        for k in (1, 5, 64):
            top = gc.decision_topk(lbs, ubs, duals, pin, [q.tolist() for q in primals], layers, init_mask, k)
            assert top[0] == dec and len(top) == min(k, n_cand)
            assert len({tuple(t) for t in top}) == len(top)
    init_mask = [torch.ones(n, dtype=torch.int32) for n in fr.net.hidden_sizes]
    with pytest.raises(RuntimeError):
        gc.decision_topk(lbs, ubs, duals, pin, [q.tolist() for q in primals], layers, init_mask, 4)


# ---- strong branching in FrontierStep ----

def _step_setup(arch='base', **kw):
    from gnn_branching_b200 import FrontierStep
    net, lbs, ubs, wp, bp = load_root(arch)
    x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))[f'{arch}_x'].copy()).reshape(-1)
    model = GraphNet(2, 64, math='tc')
    model.load_state_dict(load_gnn('random'))
    model = model.eval().cuda()
    fs = FrontierStep(model, net, x, 0.145, wp, bp, capacity=8192, decision_bound=float('inf'), **kw)
    fs.seed_root(lbs, ubs)
    return fs, (net, lbs, ubs, wp, bp, x)


def _watch(fs):
    """Record the parents every step picks and the children (with their keep flags) it adds."""
    log = {}
    pick, add = fs.queue.pick, fs.queue.add

    def pick_(*a, **kw):
        log['parents'] = pick(*a, **kw)
        return log['parents']

    def add_(d, keep=None):
        log['children'], log['keep'] = d, keep
        return add(d, keep=keep)
    fs.queue.pick, fs.queue.add = pick_, add_
    return log


def _queue_contents(fs):
    q = fs.queue.pick(len(fs.queue), float('inf'))
    out = [q.lower_bound, q.upper_bound, q.mask, q.decision] + list(q.lb) + list(q.ub)
    fs.queue.add(q)
    return [t.clone() for t in out]


def test_strong_branching_defaults_leave_the_step_unchanged():
    a, _ = _step_setup()
    b, _ = _step_setup(strong_branching_k=1, strong_branching_kw_k=0)
    assert not b.strong
    for B in (1, 2, 4, 8, 16, 32):
        sa, sb = a.step(B), b.step(B)
        assert sa == sb and sb.sb_bounded == 0 and sb.sb_changed == 0
        for x, y in zip(_queue_contents(a), _queue_contents(b)):
            assert torch.equal(x, y)
    assert b.last_strong is None


def test_strong_branching_rank0_is_the_stored_decision():
    """Scoring is batch-invariant: the parents re-scored in a batch give the decision stored when each was added alone or with
    other siblings."""
    fs, _ = _step_setup(strong_branching_k=4)
    log = _watch(fs)
    for B in (1, 2, 8, 32, 64):
        st = fs.step(B)
        cand, imp, chosen = fs.last_strong
        assert st.picked == log['parents'].B == cand.shape[0]
        assert torch.equal(cand[:, 0], log['parents'].decision), B


def test_strong_branching_first_step_against_oracle():
    from oracle import kw_bounds_oracle as KW
    fs, (net, lbs, ubs, wp, bp, x) = _step_setup(strong_branching_k=4)
    L = net.L
    st = fs.step(1)
    assert st.picked == 1 and st.added == 2
    cand, imp, chosen = fs.last_strong
    decs = [d for d in cand[0].tolist() if d[0] >= 0]
    assert len(decs) == 4
    plb = float(lbs[L + 1])

    def improvement(dec):
        lows = []
        for side in (0, 1):
            ol, ou, _ = KW.child_bounds(net, x, 0.145, wp, bp, lbs, ubs, dec, side)
            lo = float(ol[L + 1])
            lows.append(0.0 if lo > float(ou[L + 1]) else min(lo, 0.0))
        return (lows[0] + lows[1] - 2 * plb) / (-2 * plb)
    imps = [improvement(d) for d in decs]
    best = max(range(len(decs)), key=lambda r: (imps[r], -r))            # strict argmax, earliest rank on ties
    accept = {r for r in range(len(decs)) if imps[best] - imps[r] <= 1e-5}
    got = int(chosen[0])
    assert got in accept, (imps, got)
    want = decs[got]
    kids = fs.queue.pick(2, float('inf'))
    sides = {0 if float(kids.ub[want[0] + 1][i, want[1]]) == 0.0 else (1 if float(kids.lb[want[0] + 1][i, want[1]]) == 0.0 else -1)
             for i in range(2)}
    assert sides == {0, 1}, (want, sides)
    assert st.sb_bounded == 3 and st.sb_changed == int(got != 0)


@pytest.mark.parametrize('kw_k', [0, 2])
def test_strong_branching_batched_steps(kw_k):
    fs, _ = _step_setup(strong_branching_k=4, strong_branching_kw_k=kw_k)
    log = _watch(fs)
    glb, size = fs.queue.global_lb, 1
    changed = 0
    for B in (1, 2, 4, 8, 16, 32, 64, 128):
        st = fs.step(B)
        size += st.added - st.picked
        assert len(fs.queue) == size and st.children == 2 * st.picked, (st, size)
        assert st.global_lb >= glb - 1e-6
        glb = st.global_lb
        assert 0 <= st.sb_changed <= st.picked and st.sb_bounded <= st.picked * (3 + kw_k)
        changed += st.sb_changed
        cand, imp, chosen = fs.last_strong
        assert cand.shape == (st.picked, 4 + kw_k, 2)
        ar = torch.arange(st.picked, device='cuda')
        assert bool((imp[ar, chosen] >= imp[:, 0]).all())
        # no kept child's lower bound is below its parent's
        plow = log['parents'].lower_bound.repeat_interleave(2)
        keep = log['keep']
        assert bool((log['children'].lower_bound[keep] >= plow[keep] - 1e-6).all())
    assert changed > 0


def test_strong_branching_excludes_the_threshold_rule():
    with pytest.raises(ValueError):
        _step_setup(strong_branching_k=2, kw_fallback=True)
    with pytest.raises(ValueError):
        _step_setup(strong_branching_kw_k=1, kw_fallback=True)
