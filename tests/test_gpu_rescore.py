"""Option "rescore": subdomains whose activations leave the tensor-core path's fp16 operand range (|x| >= 524 288, a NaN in an
embedding) are scored again in exact fp32 on the GPU and written over the tensor-core results; every other subdomain keeps
its tensor-core result bit for bit.

Each overflow case first shows that it is one: without the option the call reports GNNB_ERR_NAN, and the exact-fp32 SIMT
mode scores the same rows finitely.  The re-scored rows must then equal the SIMT mode's rows bit for bit (the SIMT schedule
is batch-invariant) and the oracle within 1e-5 of the row's largest score.
"""
import ctypes as C
import functools

import pytest
import torch

from golden_io import ARCHS, load_gnn, load_root
from gnn_branching_b200 import GraphNet, Scorer, synthetic_frontier, _lib
from oracle import graphnet_oracle as O

pytestmark = pytest.mark.gpu

ROWS = [2, 17, 40, 63]          # the subdomains pushed out of range, spread over a 64-subdomain frontier
FACTORS = [1e6, 1e7, 1e8, 1e9, 1e10]


def _model(weights, net, math='tc', chunk=0, rescore=False, fuse=1):
    """The Scorer of a GraphNet built with the `rescore` keyword, with the network of `net` uploaded."""
    model = GraphNet(2, 64, math=math, chunk=chunk, rescore=rescore)
    model.load_state_dict(load_gnn(weights))
    model = model.eval().cuda()
    sc = model.scorer(0)
    sc.set_network(net, key=net.key)
    if math == 'tc':
        sc.set_option('fuse', fuse)
    return model, sc


def _scaled(arch, how, factor, B=64):
    """Seeded base frontier with the duals (how = 'dual') or the input box (how = 'input') of ROWS scaled by `factor`."""
    net, lbs, ubs, wp, bp = load_root(arch)
    fr = synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=4000 + ARCHS.index(arch), device='cpu')
    r = torch.tensor(ROWS)
    if how == 'dual':
        for d in fr.dual:
            d[r] *= factor
    else:
        for t in (fr.lb[0], fr.ub[0], fr.primal_input):
            t[r] *= factor
    return fr


def _score(sc, fr, dense=True):
    best, idx, scores = sc.score(fr, return_scores=dense, check=False)
    torch.cuda.synchronize()
    return best, idx, scores


def _nan_status(sc):
    """(status, NaN count) of gnnb_check: the sticky NaN report of the last DEVICE call."""
    n = C.c_int64(0)
    st = sc.lib.gnnb_check(sc.h, C.c_void_p(torch.cuda.current_stream().cuda_stream), C.byref(n))
    return st, n.value


@functools.lru_cache(maxsize=None)
def _case(arch, weights, how, fuse):
    """The overflow case and its yardsticks: the smallest factor in FACTORS for which the tensor-core pass reports NaN and the
    SIMT mode stays finite on ROWS; the option-off tensor-core outputs (written also when the call reports NaN), the SIMT outputs
    and the oracle's scores of ROWS."""
    net = load_root(arch)[0]
    _, tc = _model(weights, net, fuse=fuse)
    _, simt = _model(weights, net, math='simt')
    for f in FACTORS:
        fr = _scaled(arch, how, f)
        off = _score(tc, fr.to('cuda'))
        st, n_nan = _nan_status(tc)
        if st != _lib.GNNB_ERR_NAN:
            continue
        ref = _score(simt, fr.to('cuda'))
        assert _nan_status(simt)[0] == _lib.GNNB_OK
        if not bool(torch.isfinite(ref[2][ROWS]).all()):
            continue
        s_or, _ = O.gnn_forward(load_gnn(weights), fr._map(lambda t: t[ROWS].contiguous()))
        return dict(fr=fr, factor=f, off=off, simt=ref, oracle=s_or)
    pytest.fail(f'{arch}/{weights}/{how}: no factor in {FACTORS} overflows the tensor-core path with a finite fp32 result')


def _check_rescored(c, best, idx, scores):
    """ROWS equal the SIMT mode's results; every other row equals the option-off tensor-core results."""
    fr, (b_off, i_off, s_off), (b_ref, i_ref, s_ref) = c['fr'], c['off'], c['simt']
    best, idx = best.cuda(), idx.cuda()
    B = fr.B
    keep = torch.ones(B, dtype=torch.bool, device='cuda')
    keep[ROWS] = False
    assert torch.equal(best[keep], b_off[keep]) and torch.equal(idx[keep], i_off[keep])
    assert torch.equal(best[ROWS], b_ref[ROWS]) and torch.equal(idx[ROWS], i_ref[ROWS])
    if scores is not None:
        scores = scores.cuda()
        assert torch.equal(scores[keep], s_off[keep])
        assert torch.equal(scores[ROWS], s_ref[ROWS])
        mask = fr.mask.cuda() != 0
        masked = torch.where(mask, scores, torch.full_like(scores, float('-inf')))
        assert torch.equal(masked.max(1).values, best)
        assert bool(mask[torch.arange(B, device='cuda'), idx.long()].all())
    mask = fr.mask[ROWS]
    s = s_ref[ROWS].cpu()
    worst = max(float((s[j] - c['oracle'][j])[mask[j] != 0].abs().max()) / float(c['oracle'][j][mask[j] != 0].abs().max())
                for j in range(len(ROWS)))
    assert worst <= 1e-5, worst


def _run(c, weights, fuse, mem, chunk, out):
    _, sc = _model(weights, c['fr'].net, chunk=chunk, rescore=True, fuse=fuse)
    assert sc.get_option('rescore') == 1
    fr = c['fr'].to('cuda') if mem == 'device' else c['fr'].pin()
    if out == 'winners':
        rec = sc.score_winners(fr)
        torch.cuda.synchronize()
        best, idx, scores = rec[:, 0].view(torch.float32), rec[:, 1], None
    else:
        best, idx, scores = sc.score(fr, return_scores=(out == 'dense'))
        assert best.is_cuda == (mem == 'device')
    assert sc.rescored == len(ROWS)
    _check_rescored(c, best, idx, scores)


@pytest.mark.parametrize('out', ['dense', 'best', 'winners'])
@pytest.mark.parametrize('chunk', [0, 16])
@pytest.mark.parametrize('mem', ['device', 'host'])
@pytest.mark.parametrize('fuse', [1, 0])
def test_overflowing_duals_are_rescored(fuse, mem, chunk, out):
    """chunk = 16: the four rows are in four different waves of the tensor-core pass and of the re-score pass."""
    _run(_case('base', 'random', 'dual', fuse), 'random', fuse, mem, chunk, out)


@pytest.mark.parametrize('fuse', [1, 0])
def test_overflowing_input_box_is_rescored(fuse):
    """The overflow starts in the input-layer kernels, which have no NaN watch of their own: it is attributed to its subdomain
    by the first hidden layer's update."""
    _run(_case('base', 'random', 'input', fuse), 'random', fuse, 'device', 0, 'dense')


@pytest.mark.parametrize('arch,weights', [('wide', 'random'), ('deep', 'random'), ('base', 'shipped')])
def test_other_networks_and_weights(arch, weights):
    _run(_case(arch, weights, 'dual', 1), weights, 1, 'device', 0, 'dense')


def test_genuine_nan_is_still_reported():
    """A subdomain that is NaN in exact fp32 too (l = u = 0: 0/0 in compute_ratio, graph_conv.py:502, where the reference stops
    in pdb) is re-scored with the others and still reported; the overflow rows are right and the context stays usable."""
    c = _case('base', 'random', 'dual', 1)
    fr = c['fr']._map(lambda t: t.clone())
    fr.lb[1][5, 3] = 0.0
    fr.ub[1][5, 3] = 0.0
    _, sc = _model('random', fr.net, rescore=True)
    best, idx, scores = _score(sc, fr.to('cuda'))
    assert sc.rescored == len(ROWS) + 1
    st, n_nan = _nan_status(sc)
    assert st == _lib.GNNB_ERR_NAN and n_nan > 0
    assert torch.equal(scores[ROWS], c['simt'][2][ROWS]) and torch.equal(idx[ROWS], c['simt'][1][ROWS])
    b2, i2, s2 = sc.score(c['fr'].to('cuda'))          # raises if the NaN report or a flag were left behind
    assert sc.rescored == len(ROWS)
    _check_rescored(c, b2, i2, s2)


def test_clean_frontier_is_unchanged():
    """Base x 1 024 without overflow: the option changes no output bit and adds no kernel launch."""
    net, lbs, ubs, wp, bp = load_root('base')
    fr = synthetic_frontier(net, lbs, ubs, wp, bp, 1024, seed=2000, device='cuda')
    _, off = _model('random', net)
    _, on = _model('random', net, rescore=True)
    outs, deltas = [], []
    for sc in (off, on):
        sc.score(fr)                                       # warm-up: workspace and buffers
        n0 = sc.launches
        outs.append(sc.score(fr))
        deltas.append(sc.launches - n0)
    assert on.rescored == 0 and off.rescored == 0
    assert deltas[0] == deltas[1]
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    rec_off, rec_on = off.score_winners(fr), on.score_winners(fr)
    torch.cuda.synchronize()
    assert torch.equal(rec_off, rec_on)
    # the exact-fp32 mode accepts the option and has nothing to re-score
    simt = Scorer(0, math='simt', rescore=True)
    simt.set_gnn(load_gnn('random'))
    simt.set_network(fr.net)
    simt.score(fr.slice(0, 8).contiguous())
    assert simt.get_option('rescore') == 1 and simt.rescored == 0
