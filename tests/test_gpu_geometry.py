"""Every device entry point on networks whose geometry takes the branches the CIFAR nets never reach.

The kernels branch on the shape of the verified network: how a layer is cut into 128-slot tiles (grid tiles, range tiles
for 1x1 maps, channel blocks past 128), whether a conv layer's KW bounds take the windowed cone kernel (and its 8-column
vector loop or its scalar loop) or the dense recursion, how many hidden layers there are (one: the first hidden layer is
also the last), and how many taps of conv_transpose2d reach an input position.  The catalogue below has one small seeded
network per branch; ``_assert_branch`` restates the host-side rule that sends it there (tile counts, the cone kernel's
qualification rule with its 200 KB window formula, layer counts, tap counts), so that a later change to a limit fails
loudly instead of letting a test pass without reaching its branch.

Scoring, top-k, BaBSR, gradients and the domain queue run in the pytest process; the KW bound checks, FrontierStep and the
size limits run in their own process (``_run_isolated``: python tests/test_gpu_geometry.py <check> <arg>, exit code 0 =
pass).
"""
import functools
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import pytest                                                    # noqa: E402
import torch                                                     # noqa: E402
from torch import nn                                             # noqa: E402

from golden_io import load_gnn                                   # noqa: E402
from gnn_branching_b200 import Flatten, netspec_from_modules, synthetic_frontier      # noqa: E402
from oracle import graphnet_oracle as O                          # noqa: E402
from oracle import kw_bounds_oracle as KW                        # noqa: E402

RTOL = {'simt': 1e-5, 'tc': 1e-4}
KW_TOL = 5e-5                   # KW bounds: max|got - want| <= KW_TOL * max(1, max|want|) per layer
BABSR_RTOL = 1e-5
GRAD_RTOL = 2e-2                # the batched gradient tolerance of test_gpu_parity (ReLU masks that flip between fp32 evaluations)
B_SCORE = 64

# the library's limits, restated (gnnb_prop_tc.cu, gnnb_kw.cu, gnnb_queue.cu, gnnb_babsr.cu, gnnb_api.cu)
TILE = 128
CONE_MAX_DEPTH, CONE_MAX_COLS, CONE_MAX_SMEM = 8, 256, 200 * 1024
QUEUE_MAX_LAYERS, KW_MAX_LAYERS, BABSR_MAX_LAYERS = 16, 30, 32
CONV_WEIGHT_MAX_BYTES = 64 * 1024


# ---- the catalogue -----------------------------------------------------------------------------------------------------
def _conv(ci, co, k, s, p):
    return [nn.Conv2d(ci, co, k, stride=s, padding=p), nn.ReLU()]


def _lin(i, o):
    return [nn.Linear(i, o), nn.ReLU()]


# name: (fixed layers, input shape, eps).  eps is raised from 0.05 where the root has too few ambiguous ReLUs for a frontier
# with candidates in every subdomain (one_conv, one_linear) or where no child then takes the second KW pass (pointwise_out,
# wide_cone, gap_first); on big_cone, stride3 and tile_edges no split takes it at any eps tried (up to 0.5).  An optional fourth
# entry is the conv weights' standard deviation (default 0.3): at 0.3 the 600-tap windows of big_cone drive the GNN's
# embeddings past the fp16 operand range of the tensor-core mode (GNNB_ERR_NAN, see option "rescore").
CATALOGUE = {
    'one_conv': (lambda: _conv(1, 3, 3, 2, 1), (1, 7, 7), 0.2),
    'one_linear': (lambda: [Flatten()] + _lin(10, 7), (1, 1, 10), 1.0),
    'tile_edges': (lambda: _conv(2, 129, 3, 1, 1) + [Flatten()] + _lin(516, 129) + _lin(129, 1), (2, 2, 2), 0.05),
    'pointwise_out': (lambda: _conv(3, 130, 4, 1, 0) + _conv(130, 20, 1, 1, 0) + [Flatten()] + _lin(20, 5), (3, 4, 4), 0.2),
    'wide_cone': (lambda: _conv(2, 4, 3, 1, 1) + _conv(4, 260, 3, 1, 1) + [Flatten()] + _lin(4160, 10), (2, 4, 4), 0.5),
    'nine_convs': (lambda: _conv(1, 4, 3, 1, 1) + sum([_conv(4, 4, 3, 1, 1) for _ in range(8)], []) + [Flatten()] + _lin(100, 6),
                   (1, 5, 5), 0.05),
    'big_cone': (lambda: _conv(3, 24, 5, 1, 2) + _conv(24, 24, 5, 1, 2) + _conv(24, 24, 5, 1, 2) + [Flatten()] + _lin(3456, 8),
                 (3, 12, 12), 0.05, 0.1),
    'stride3': (lambda: _conv(2, 6, 5, 3, 2) + _conv(6, 7, 3, 1, 1) + [Flatten()] + _lin(84, 3), (2, 10, 7), 0.05),
    'gap_first': (lambda: _conv(2, 4, 1, 2, 0) + _conv(4, 6, 3, 1, 1) + [Flatten()] + _lin(96, 5), (2, 7, 7), 0.2),
    'gap_hidden': (lambda: _conv(2, 4, 3, 1, 1) + _conv(4, 5, 1, 2, 0) + [Flatten()] + _lin(80, 6), (2, 7, 7), 0.05),
}
NAMES = list(CATALOGUE)
SCORED = [n for n in NAMES if n != 'gap_hidden']          # gap_hidden: the GNN scoring entries refuse it


@functools.lru_cache(maxsize=None)
def _net(name):
    """(net, x, wp, bp, eps): conv / linear weights ~ N(0, 0.3^2), biases ~ N(0, 0.1^2), x ~ N(0, 1), wp ~ N(0, 0.3^2)."""
    make, shape, eps, wstd = (CATALOGUE[name] + (0.3,))[:4]
    layers = make()
    g = torch.Generator().manual_seed(1000 + NAMES.index(name))
    for m in layers:
        for q in m.parameters():
            q.requires_grad = False
            q.data = torch.randn(q.shape, generator=g) * ((wstd if q.dim() == 4 else 0.3) if q.dim() > 1 else 0.1)
    net = netspec_from_modules(layers, shape, name=name)
    x = torch.randn(shape, generator=g).reshape(-1)
    wp = torch.randn(net.hidden_sizes[-1], generator=g) * 0.3
    return net, x, wp, 0.1, eps


@functools.lru_cache(maxsize=None)
def _root(name):
    """KW root bounds of the net's (x, wp, bp) (the bounds part of build_the_model)."""
    net, x, wp, bp, eps = _net(name)
    return KW.root_bounds(net, x, eps, wp, bp)


@functools.lru_cache(maxsize=None)
def _frontier(name, B=B_SCORE, seed=7):
    net, x, wp, bp, eps = _net(name)
    lbs, ubs = _root(name)
    return synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=seed, max_splits=4)


# ---- the branches, restated --------------------------------------------------------------------------------------------
def _grid_tiles(C, H, W):
    """gnnb_prop_tc.cu grid_tiles: the (Yb, Xb) spatial block with the fewest tiles, channel blocks of up to 128."""
    Cb = min(C, TILE)
    Pp = max(1, TILE // Cb)
    best = None
    for yb in range(1, min(H, Pp) + 1):
        for xb in range(1, min(W, Pp // yb) + 1):
            t = (-(-H // yb)) * (-(-W // xb))
            if best is None or t < best[0] or (t == best[0] and abs(yb - xb) < abs(best[1] - best[2])):
                best = (t, yb, xb)
    return -(-C // Cb) * best[0]


def _tiles(net, k):
    """Tiles of layer k (0 = input): range tiles of 128 nodes for 1x1 maps and linear layers, grid tiles otherwise
    (make_tiling)."""
    C, H, W = net.input_shape if k == 0 else (tuple(net.affine[k - 1].out_shape) + (1, 1))[:3]
    if H == 1 and W == 1:
        return -(-C // TILE), 'range'
    return _grid_tiles(C, H, W), 'grid'


def _cone(net, k):
    """kw_cone_layer's rule for the bounds of hidden layer k (1-based): (qualifies, reason, vector loop)."""
    if k < 2:
        return False, 'first layer', False
    if k > CONE_MAX_DEPTH:
        return False, 'depth', False
    if any(net.affine[j].kind != 'conv' for j in range(k)):
        return False, 'linear in front', False
    cols = net.affine[k - 1].out_shape[0]
    if cols > CONE_MAX_COLS:
        return False, 'columns', False
    R = max(1, 256 // cols)
    h = w = 1
    max_elems = 0
    for j in range(k, 0, -1):
        a = net.affine[j - 1]
        ks = a.weight.shape[2]
        h = min((h - 1) * a.stride + ks, a.in_shape[1])
        w = min((w - 1) * a.stride + ks, a.in_shape[2])
        max_elems = max(max_elems, a.in_shape[0] * h * w)
    smem = 2 * max(max_elems * cols, 5 * cols * R) * 4
    if smem > CONE_MAX_SMEM:
        return False, 'window', False
    return True, 'cone', cols % 8 == 0


def _axis_taps(i, k, s, p, n_out):
    return sum(1 for t in range(k) if i + p - t >= 0 and (i + p - t) % s == 0 and (i + p - t) // s < n_out)


def _zero_tap_layers(net):
    """1-based conv layers with an input position that no tap of conv_transpose2d reaches (the host formula of k_div_freq)."""
    out = []
    for j, a in enumerate(net.affine):
        if a.kind != 'conv':
            continue
        k, s, p = a.weight.shape[2], a.stride, a.padding
        if any(_axis_taps(y, k, s, p, a.out_shape[1]) == 0 for y in range(a.in_shape[1])) or \
                any(_axis_taps(x, k, s, p, a.out_shape[2]) == 0 for x in range(a.in_shape[2])):
            out.append(j + 1)
    return out


def _assert_branch(name):
    net = _net(name)[0]
    L = net.L
    cones = {k: _cone(net, k) for k in range(1, L + 1)}
    gaps = _zero_tap_layers(net)
    if name != 'gap_first':
        assert gaps == ([2] if name == 'gap_hidden' else []), (name, gaps)
    if name == 'one_conv':
        assert L == 1 and net.affine[0].kind == 'conv'
    elif name == 'one_linear':
        assert L == 1 and net.affine[0].kind == 'linear' and net.input_shape[1:] == (1, 10)
    elif name == 'tile_edges':
        assert _tiles(net, 1) == (2 * 4, 'grid') and net.affine[0].out_shape[0] == TILE + 1      # 2 channel blocks x 4 positions
        assert _tiles(net, 2) == (2, 'range') and net.hidden_sizes[1] == TILE + 1                 # a 129-node linear layer
        assert [a.kind for a in net.affine[1:]] == ['linear', 'linear'] and net.hidden_sizes[-1] == 1
    elif name == 'pointwise_out':
        assert net.affine[0].out_shape[1:] == (1, 1) and _tiles(net, 1) == (2, 'range')          # 130 channels of a 1x1 map
        assert net.affine[1].out_shape[1:] == (1, 1) and _tiles(net, 2) == (1, 'range')
        assert cones[2] == (True, 'cone', False)                                                 # 20 columns: the scalar loop
    elif name == 'wide_cone':
        assert cones[2][:2] == (False, 'columns')
    elif name == 'nine_convs':
        assert L == 10 and all(cones[k][0] for k in range(2, 9)) and cones[9][:2] == (False, 'depth')
    elif name == 'big_cone':
        assert cones[2] == (True, 'cone', True) and cones[3][:2] == (False, 'window')
    elif name == 'stride3':
        a = net.affine[0]
        assert a.stride == 3 and a.in_shape[1] != a.in_shape[2] and a.out_shape[1] != a.out_shape[2]
        assert a.weight.shape[2] == 5 and cones[2] == (True, 'cone', False)
    elif name == 'gap_first':
        assert gaps == [1] and net.affine[0].weight.shape[2] < net.affine[0].stride
    elif name == 'gap_hidden':
        assert net.affine[1].weight.shape[2] < net.affine[1].stride


def test_catalogue_reaches_its_branches():
    """Host-side only: every network of the catalogue builds and takes the branch it is there for, and the oracle's scores
    of a small frontier are finite, except behind the zero-tap layer of gap_hidden, where the reference divides 0 by 0."""
    sd = load_gnn('random')
    for name in NAMES:
        _assert_branch(name)
        fr = _frontier(name, 2, seed=3)
        assert bool((fr.mask != 0).any(1).all()), (name, 'a subdomain without candidates')
        s, _ = O.gnn_forward(sd, fr)
        assert bool(torch.isfinite(s).all()) == (name != 'gap_hidden'), name
        if name != 'gap_hidden':
            assert _oracle_scores(name)[1] < 5e-5, (name, 'the float32 oracle is far from the float64 one')


# ---- scoring -----------------------------------------------------------------------------------------------------------
def _scorer(net, math, fuse=1, chunk=0):
    from test_gpu_mixed_batches import _scorer as make
    return make(net, math, chunk, fuse)


def _f64(fr, sd):
    """The frontier, its network and the GNN parameters in float64."""
    import copy
    net = copy.deepcopy(fr.net)
    for a in net.affine:
        a.weight, a.bias = a.weight.double(), a.bias.double()
    f = fr._map(lambda t: t.double())
    f.net = net
    return f, {k: v.detach().double().clone() for k, v in sd.items()}


def _row_rel(a, b, mask):
    m = mask != 0
    d = torch.where(m, (a.double() - b.double()).abs(), torch.zeros_like(b, dtype=torch.float64)).amax(1)
    s = torch.where(m, b.double().abs(), torch.zeros_like(b, dtype=torch.float64)).amax(1)
    return float((d / s.clamp(min=1e-300)).max())


@functools.lru_cache(maxsize=None)
def _oracle_scores(name, kind='synthetic'):
    """(scores of the oracle evaluated in float64, conditioning): the kernels are held to the float64 evaluation with their
    mode's tolerance plus twice the distance of the oracle's own float32 evaluation from it (up to 2.7e-5 of the row maximum on
    these nets: 129-wide and 4160-wide sums, all-ambiguous layers; about 1e-6 on the CIFAR nets)."""
    fr = _frontier(name) if kind == 'synthetic' else _decided(name, kind)
    sd = load_gnn('random')
    s32, _ = O.gnn_forward(sd, fr)
    f, sd64 = _f64(fr, sd)
    with torch.no_grad():
        s64, _ = O.gnn_forward(sd64, f, keep_graph=True)
    m = fr.mask != 0
    assert bool(torch.isfinite(s64[m]).all()), (name, kind)
    return s64.detach(), _row_rel(s32, s64, fr.mask)


def _score_and_check(name, fr, oracle, what):
    """gnnb_score in every mode against the oracle, fuse 1 against fuse 0, host against device buffers, gnnb_score_topk against
    the dense scores of the same call."""
    from gpu_isolated import _close
    from test_gpu_mixed_batches import _bits, _same, _score
    from test_gpu_topk import _ref_topk
    net = fr.net
    mask = fr.mask.cuda()
    s_or, cond = oracle
    got = {}
    for math, fuse in (('tc', 1), ('tc', 0), ('simt', 1)):
        sc = _scorer(net, math, fuse)
        best, idx, scores = ref = _score(sc, fr, 'device')
        rep = O.parity_report(scores.cpu(), s_or, fr.mask, idx.cpu(), rtol=RTOL[math] + 2 * cond)
        assert rep['ok'] and rep['decisions_checked'] >= fr.B // 2, (what, math, fuse, cond, rep)
        m = mask != 0
        assert torch.equal(torch.where(m, scores, torch.full_like(scores, float('-inf'))).max(1).values, best), (what, math, fuse)
        assert _same(_score(sc, fr, 'host'), ref), (what, math, fuse, 'host buffers')
        ts, ti, s2 = sc.score_topk(fr.to('cuda'), 5, return_scores=True)
        torch.cuda.synchronize()
        assert torch.equal(_bits(s2), _bits(scores)), (what, math, fuse, 'top-k call, dense scores')
        assert torch.equal(_bits(ts[:, 0]), _bits(best)) and torch.equal(ti[:, 0], idx), (what, math, fuse, 'top-k column 0')
        rs, ri = _ref_topk(scores, mask, 5)
        assert torch.equal(_bits(ts), _bits(rs)) and torch.equal(ti, ri), (what, math, fuse, 'top-k order')
        got[(math, fuse)] = ref
    (b1, i1, s1), (b0, i0, s0) = got[('tc', 1)], got[('tc', 0)]
    _close(s0, s1, i0, i1, mask, f'{what}: fuse 0 vs 1', rtol=1e-5 + 2 * cond)      # accumulation order, as against the oracle


@pytest.mark.gpu
@pytest.mark.parametrize('name', SCORED)
def test_scores_match_oracle(name):
    _assert_branch(name)
    _score_and_check(name, _frontier(name), _oracle_scores(name), name)


# ---- frontiers with a decided layer ----------------------------------------------------------------------------------
def _base_net():
    from golden_io import load_root
    net, lbs, ubs, wp, bp = load_root('base')
    return net, lbs, ubs, wp, bp


@functools.lru_cache(maxsize=None)
def _decided(name, kind):
    """kind 'dead': every node of the second hidden layer has l >= 0 or u <= 0 in every subdomain (its ambiguous nodes are
    fixed to a seeded side, as a split does), so the layer has no ambiguous row; 'all_amb': every node of the first hidden
    layer is ambiguous in every subdomain."""
    if name == 'base':
        net, lbs, ubs, wp, bp = _base_net()
        fr = synthetic_frontier(net, lbs, ubs, wp, bp, B_SCORE, seed=17, max_splits=32)
    else:
        fr = _frontier(name, B_SCORE, seed=17)
    fr = fr._map(lambda t: t.clone())
    g = torch.Generator().manual_seed(23)
    k = 2 if kind == 'dead' else 1
    lb, ub = fr.lb[k], fr.ub[k]
    if kind == 'dead':
        amb = (lb < 0) & (ub > 0)
        up = torch.rand(lb.shape, generator=g) < 0.5
        lb[amb & up] = 0.0
        ub[amb & ~up] = 0.0
    else:
        lb.copy_(torch.minimum(lb, -0.05 - 0.1 * torch.rand(lb.shape, generator=g)))
        ub.copy_(torch.maximum(ub, 0.05 + 0.1 * torch.rand(ub.shape, generator=g)))
    amb = ((lb < 0) & (ub > 0)).float()
    fr.dual[k - 1] *= amb.unsqueeze(-1)
    off = sum(fr.net.hidden_sizes[:k - 1])
    fr.mask[:, off:off + fr.net.hidden_sizes[k - 1]] = amb
    if kind == 'dead':
        assert not bool(amb.any()) and bool((fr.mask != 0).any(1).all())
    else:
        assert bool(amb.all())
    return fr


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['dead', 'all_amb'])
@pytest.mark.parametrize('name', ['base', 'tile_edges'])
def test_decided_layers_match_oracle(name, kind):
    """A hidden layer without a single ambiguous row in any subdomain (the ambiguous-row compaction and the relaxation kernels
    see zero rows), and a first hidden layer that is ambiguous everywhere: scoring and BaBSR against the oracles."""
    if name != 'base':
        _assert_branch(name)
    fr = _decided(name, kind)
    _score_and_check(name, fr, _oracle_scores(name, kind), f'{name} {kind}')
    _babsr_and_check(fr, f'{name} {kind}')


# ---- BaBSR -------------------------------------------------------------------------------------------------------------
def _babsr_safe(s_or, ic, mask, sizes, tol, branch):
    """Rows whose oracle decision no perturbation within ``tol`` can change, per branch of the decision rule."""
    B = s_or.shape[0]
    offs = [0]
    for n in sizes:
        offs.append(offs[-1] + n)
    safe = torch.ones(B, dtype=torch.bool)
    if branch == 'score':
        top2 = s_or.topk(min(2, s_or.shape[1]), dim=1).values
        safe &= (top2[:, 0] - top2[:, -1]) > 2 * tol
        safe &= (top2[:, 0] - 0.001).abs() > 2 * tol
        for k in range(len(sizes)):                       # the in-layer maxima decide the layer
            t = s_or[:, offs[k]:offs[k + 1]].topk(min(2, sizes[k]), dim=1).values
            safe &= ((t[:, 0] - top2[:, 0]).abs() > 2 * tol) | (t[:, 0] == top2[:, 0])
    if branch in ('score', 'intercept'):
        for k in range(len(sizes)):
            lay = ic[:, offs[k]:offs[k + 1]]
            low = lay.topk(min(2, sizes[k]), dim=1, largest=False).values
            safe &= (low[:, 0] + 1e-4).abs() > 2 * tol
            if sizes[k] > 1:
                safe &= ((low[:, 1] - low[:, 0]) > 2 * tol) | (low[:, 0] >= -1e-4 + 2 * tol)
    return safe


def _babsr_and_check(fr, what):
    """gnnb_babsr in the three branches of the decision rule (threshold, then intercept, then preference order) against the
    oracle: scores within 1e-5 of the largest oracle score, decisions, counters and kinds wherever the oracle's decision is
    safe from rounding; host buffers give the device results."""
    from gnn_branching_b200 import Scorer
    from oracle import babsr_oracle as BO
    net = fr.net
    L = net.L
    order = [0] + [k for k in range(L) if k != 0]
    sc = Scorer(0)
    sc.set_network(net, key=net.key)
    s_or, ic = BO.babsr_scores(fr)
    tol = BABSR_RTOL * float(s_or.abs().max())
    for branch, (thr, cnt) in {'score': (0.001, 0), 'intercept': (1e9, 0), 'order': (1e9, 2)}.items():
        counters = [cnt] * fr.B
        dec, cout, kind, scores = sc.babsr(fr.to('cuda'), counters, order, 0, thr, return_scores=True)
        torch.cuda.synchronize()
        assert float((scores.cpu() - s_or).abs().max()) <= tol, (what, branch)
        d_or, c_or, k_or = BO.babsr_decide(s_or, ic, fr.mask, net.hidden_sizes, counters, order, 0, thr)
        safe = _babsr_safe(s_or, ic, fr.mask, net.hidden_sizes, tol, branch)
        assert int(safe.sum()) >= fr.B // 8, (what, branch, int(safe.sum()))
        assert torch.equal(dec.cpu()[safe].long(), d_or[safe]), (what, branch, 'decisions')
        assert torch.equal(cout.cpu()[safe].long(), c_or[safe]) and torch.equal(kind.cpu()[safe].long(), k_or[safe]), (what, branch)
        d2, c2, k2, s2 = sc.babsr(fr, counters, order, 0, thr, return_scores=True)
        assert torch.equal(d2, dec.cpu()) and torch.equal(c2, cout.cpu()) and torch.equal(k2, kind.cpu()) and torch.equal(s2, scores.cpu())


@pytest.mark.gpu
@pytest.mark.parametrize('name', NAMES)
def test_babsr_matches_oracle(name):
    _assert_branch(name)
    _babsr_and_check(_frontier(name), name)


# ---- the zero-tap geometry -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_zero_tap_hidden_layer_is_refused_by_the_gnn_entries():
    """gap_hidden: conv_transpose2d of its second conv layer (1x1 kernel, stride 2) reaches no input position of odd
    coordinates, and the GNN's backward propagation divides those by a tap count of 0 (NaN scores in the reference).  Both math
    modes, top-k, winner records and gradients refuse the network with GNNB_ERR_UNSUPPORTED, naming the layer; the context
    then still scores gap_first."""
    from gnn_branching_b200 import _lib
    from test_gpu_mixed_batches import _terms
    _assert_branch('gap_hidden')
    fr = _frontier('gap_hidden')
    net = fr.net
    fd = fr.to('cuda')
    for math in ('tc', 'simt'):
        sc = _scorer(net, math)
        for call in (lambda: sc.score(fd), lambda: sc.score(fr), lambda: sc.score_topk(fd, 5), lambda: sc.score_winners(fd),
                     lambda: sc.score_grad(fd.slice(0, 2).contiguous(), _terms(fr.slice(0, 2)))):
            with pytest.raises(_lib.GnnbError) as ei:
                call()
            assert ei.value.status == _lib.GNNB_ERR_UNSUPPORTED and 'layer 2' in str(ei.value), (math, str(ei.value))
        other = _frontier('gap_first')
        sc.set_network(other.net, key=other.net.key)
        _, idx, scores = sc.score(other.to('cuda'))
        s_or, cond = _oracle_scores('gap_first')
        rep = O.parity_report(scores.cpu(), s_or, other.mask, idx.cpu(), rtol=RTOL[math] + 2 * cond)
        assert rep['ok'], (math, rep)


# ---- gradients ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('name', SCORED)
def test_score_grad_matches_oracle(name):
    """gnnb_score_grad on 3 subdomains: term scores within 1e-5 and gradients within the batched tolerance of the float64 autograd
    oracle; the batched forward is batch invariant (term scores equal single-domain calls bit for bit) and the batched gradient
    is the sum of the single-domain gradients up to the order of the atomicAdds."""
    from test_gpu_mixed_batches import _bits, _terms
    from test_gpu_parity import _assert_grads
    _assert_branch(name)
    fr = _frontier(name).slice(0, 3).contiguous()
    terms = _terms(fr)
    ref, vals_ref = _score_grads64(fr, terms)
    sc = _scorer(fr.net, 'tc')
    fd = fr.to('cuda')
    vals = sc.score_grad(fd, terms)
    assert float((vals - vals_ref).abs().max()) <= 1e-5 * float(vals_ref.abs().max()), name
    g = sc.gradients()
    _assert_grads(g, ref, rtol=GRAD_RTOL)
    singles, single_vals = [], []
    for b in range(fr.B):
        single_vals.append(sc.score_grad(fd.slice(b, b + 1).contiguous(), [(0, i, cf) for d, i, cf in terms if d == b]))
        singles.append(sc.gradients())
    assert torch.equal(_bits(vals), _bits(torch.cat(single_vals))), (name, 'the batched forward is not batch invariant')
    for k in g:
        tol = 1e-5 * sum(float(s[k].abs().max()) for s in singles)
        err = float((g[k] - sum(s[k] for s in singles)).abs().max())
        assert err <= tol, (name, k, err, tol)


def _score_grads64(fr, terms):
    """online_oracle.score_grads evaluated in float64 (autograd through the oracle's forward)."""
    f, params = _f64(fr, load_gnn('random'))
    for v in params.values():
        v.requires_grad_(True)
    scores, _ = O.gnn_forward(params, f, keep_graph=True)
    sum(c * scores[b, i] for b, i, c in terms).backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)).detach().float() for k, v in params.items()}
    return grads, torch.stack([scores[b, i] for b, i, _ in terms]).detach().float()


# ---- domain queue ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('name', ['one_conv', 'nine_convs'])
def test_domain_queue_round_trip(name):
    """Batched adds with a keep mask, picks and prunes against the queue oracle; every picked domain's payload (bounds of every
    layer, mask, decision) comes back bit for bit."""
    from gnn_branching_b200 import DomainQueue, Scorer
    from oracle.queue_oracle import QueueOracle
    from test_gpu_parity import _check_payload, _queue_batch
    _assert_branch(name)
    net = _net(name)[0]
    sc = Scorer(0)
    sc.set_network(net, key=net.key)
    q, o = DomainQueue(sc, capacity=400), QueueOracle()
    g = torch.Generator().manual_seed(9)
    nid = 0
    for rnd in range(6):
        B = 90
        lbs = (torch.round(torch.randn(B, generator=g) * 8) / 8 - 1.0).tolist()
        keep = torch.rand(B, generator=g) < 0.7
        ids = list(range(nid, nid + B))
        nid += B
        assert q.add(_queue_batch(net, lbs, ids), keep=keep.cuda()) == int(keep.sum())
        for b in range(B):
            if keep[b]:
                o.add(lbs[b], ids[b])
        assert len(q) == len(o.domains) and q.global_lb == o.domains[0].lower_bound
        thr = float(torch.randn(1, generator=g)) * 0.5 - 0.8
        want = []
        for _ in range(50):
            if not o.domains or o.domains[0].lower_bound >= thr:
                break
            want.append(o.pick(thr))
        b = q.pick(50, thr)
        assert [int(x) // 2 for x in b.decision[:, 1].cpu()] == want
        _check_payload(net, b, want)
        if rnd % 2 == 1:
            pt = float(torch.randn(1, generator=g)) * 0.5
            q.prune(pt)
            o.prune(pt)
        assert len(q) == len(o.domains)
    rest = q.pick(len(q), float('inf'))
    left = [i for _, i in o.state()]
    assert [int(x) // 2 for x in rest.decision[:, 1].cpu()] == left
    _check_payload(net, rest, left)


# ---- KW bounds, FrontierStep, limits (own process) ---------------------------------------------------------------------
def _iso(what, arg, timeout=300, env=None):
    from test_gpu_parity import _run_isolated
    _run_isolated(what, arg, timeout=timeout, env=env, script=os.path.basename(__file__))


# nets on which the cone kernel bounds at least one layer: the dense recursion (GNNB_KW_DENSE=1) must give the same bounds
CONE_NETS = [n for n in NAMES if any(_cone(_net(n)[0], k)[0] for k in range(2, _net(n)[0].L + 1))]


@pytest.mark.gpu
@pytest.mark.parametrize('dense', ['0', '1'])
@pytest.mark.parametrize('name', NAMES)
def test_kw_bounds_match_oracle(name, dense):
    if dense == '1' and name not in CONE_NETS:
        pytest.skip('no layer of this net takes the cone kernel: the dense recursion is the default path')
    _assert_branch(name)
    _iso('kw', name, env={'GNNB_KW_DENSE': dense})


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['one_conv', 'stride3'])
def test_frontier_step(name):
    _assert_branch(name)
    _iso('frontier_step', name)


@pytest.mark.gpu
def test_size_limits_refuse_and_leave_the_context_usable():
    _iso('limits', '-', timeout=400)


def _err(a, b):
    return float((a.reshape(-1).cpu() - b.reshape(-1)).abs().max()) / max(1.0, float(b.abs().max()))


def _check_bounds(gl, gu, i, want_l, want_u, what):
    worst = 0.0
    for k in range(len(want_l)):
        e = max(_err(gl[k][i], want_l[k]), _err(gu[k][i], want_u[k]))
        worst = max(worst, e)
        assert e <= KW_TOL, (what, i, k, e)
    return worst


def _children(name):
    """One seeded ambiguous ReLU of the root in every hidden layer that has one, both choices."""
    net = _net(name)[0]
    lbs, ubs = _root(name)
    g = torch.Generator().manual_seed(4)
    decs = []
    for lay in range(net.L):
        amb = ((lbs[lay + 1] < 0) & (ubs[lay + 1] > 0)).nonzero().view(-1)
        if amb.numel():
            i = int(amb[int(torch.randint(0, amb.numel(), (1,), generator=g))])
            decs += [(lay, i, 0), (lay, i, 1)]
    return decs


def _gain(net, x, eps, wp, bp, lbs, ubs, dec):
    """Largest relative interval gain on a hidden layer behind the split after the first KW pass: the library repeats the KW
    pass where it exceeds rounding (the rule of gpu_isolated.check_child_bounds)."""
    lay, idx, choice = dec
    lbs, ubs = [t.clone() for t in lbs], [t.clone() for t in ubs]
    (ubs if choice == 0 else lbs)[lay + 1][idx] = 0
    lbs, ubs = KW._kw_pass(net, x, eps, wp, bp, lbs, ubs, keep_upto=lay + 1)
    g = 0.0
    for k in range(lay + 2, net.L + 1):
        lo, hi = KW.interval_layer(net.affine[k - 1], lbs[k - 1].clamp(min=0), ubs[k - 1].clamp(min=0))
        g = max(g, float(((lo - lbs[k]) / lbs[k].abs().clamp(min=1)).max()), float(((ubs[k] - hi) / ubs[k].abs().clamp(min=1)).max()))
        lbs[k], ubs[k] = torch.max(lbs[k], lo), torch.min(ubs[k], hi)
    return g


def _root_moved(net, x, eps, wp, bp):
    from test_gpu_mixed_batches import _root_moved as moved
    return moved(net, x, eps, wp, bp)


def check_kw(name):
    """gnnb_kw_bounds (root, and every child's split bounds provided), gnnb_root_bounds and gnnb_child_bounds (every child in
    one batched call) against the KW oracle, math 0 and 1; the BaB masks from the bounds; the second-pass flags by the
    interval-gain rule; the root's second-pass flag by the "a hidden layer moved by more than 1e-4" rule."""
    from gnn_branching_b200 import Scorer
    net, x, wp, bp, eps = _net(name)
    L = net.L
    lbs, ubs = _root(name)
    k_l, k_u = KW.kw_bounds(net, x, eps, wp, bp)
    decs = _children(name)
    B = len(decs)
    assert B >= 2, (name, 'no ambiguous ReLU at the root')
    want = [KW.child_bounds(net, x, eps, wp, bp, lbs, ubs, d[:2], d[2]) for d in decs]
    split = [KW.split_bounds(lbs, ubs, d[:2], d[2]) for d in decs]
    want_split = [KW.kw_bounds(net, x, eps, wp, bp, *s) for s in split]
    gains = [_gain(net, x, eps, wp, bp, lbs, ubs, d) for d in decs]
    moved = _root_moved(net, x, eps, wp, bp)
    dec = torch.tensor(decs, dtype=torch.int32)
    for math in (0, 1):
        sc = Scorer(0)
        sc.set_network(net, key=net.key)
        sc.set_option('math', math)
        what = f'{name} math={math}'
        gl, gu = sc.kw_bounds(x.reshape(1, -1), eps, wp.reshape(1, -1), torch.tensor([bp]))
        w_root = _check_bounds(gl, gu, 0, k_l, k_u, (what, 'kw_bounds'))
        plb = [torch.stack([s[0][k] for s in split]) for k in range(L)]
        pub = [torch.stack([s[1][k] for s in split]) for k in range(L)]
        gl, gu = sc.kw_bounds(x.reshape(1, -1), eps, wp.reshape(1, -1).repeat(B, 1), torch.full((B,), float(bp)), plb, pub)
        for i in range(B):
            _check_bounds(gl, gu, i, *want_split[i], (what, 'kw_bounds provided'))
        rl, ru, rmask, rsecond = sc.root_bounds(x.reshape(1, -1), eps, wp.reshape(1, -1), torch.tensor([bp]))
        torch.cuda.synchronize()
        _check_bounds(rl, ru, 0, lbs, ubs, (what, 'root_bounds'))
        if not 0.5e-4 < moved < 2e-4:
            assert int(rsecond[0]) == int(moved > 1e-4), (what, 'root second pass', moved)
        gl, gu, masks, second = sc.child_bounds(x.reshape(1, -1), eps, wp.reshape(1, -1).repeat(B, 1), torch.full((B,), float(bp)),
                                                [t.reshape(1, -1).repeat(B, 1) for t in lbs], [t.reshape(1, -1).repeat(B, 1) for t in ubs],
                                                dec[:, 0], dec[:, 1], dec[:, 2])
        torch.cuda.synchronize()
        worst = 0.0
        for i, (lay, idx, choice) in enumerate(decs):
            worst = max(worst, _check_bounds(gl, gu, i, want[i][0], want[i][1], (what, 'child_bounds', decs[i])))
            if gains[i] > 1e-5 or gains[i] < 1e-7:
                assert int(second[i]) == int(gains[i] > 1e-5), (what, 'second pass', decs[i], int(second[i]), gains[i])
            if lay == L - 1:
                assert int(second[i]) == 0, (what, 'second pass behind the last hidden layer', decs[i])
            for k in range(1, L + 1):
                l, u = gl[k][i].cpu(), gu[k][i].cpu()
                m = torch.where((l >= 0) & (u >= 0), 1, torch.where((l <= 0) & (u <= 0), 0, -1)).to(torch.int8)
                assert torch.equal(masks[k - 1][i].cpu(), m), (what, 'mask', decs[i], k)
            assert int(masks[lay][i][idx]) == choice, (what, 'mask of the split node', decs[i])
        print(f'kw {what} dense={os.environ.get("GNNB_KW_DENSE", "0")}: root err {w_root:.2e}, {B} children, worst rel err '
              f'{worst:.2e}, second passes {second.tolist()}', flush=True)


def check_frontier_step(name):
    """FrontierStep on the net's root (the oracle's KW root bounds): the first step's two children carry the oracle's child
    bounds for the root's GNN decision; over 4 batched steps every child's lower bound is at least its parent's, the queue holds
    exactly the children that were kept and its global lower bound never decreases."""
    from gnn_branching_b200 import FrontierStep, GraphNet
    net, x, wp, bp, eps = _net(name)
    lbs, ubs = _root(name)
    model = GraphNet(2, 64, math='tc')
    model.load_state_dict(load_gnn('random'))
    model = model.eval().cuda()
    fs = FrontierStep(model, net, x, eps, wp, bp, capacity=8192, decision_bound=float('inf'))
    fs.seed_root(lbs, ubs)
    assert len(fs.queue) == 1
    root = fs.queue.pick(1, float('inf'))
    dec = root.decision[0].tolist()
    assert dec[0] >= 0, (name, 'the root has no branching candidate')
    fs.queue.add(root)
    st = fs.step(8)
    assert (st.picked, st.children) == (1, 2) and st.added == 2 - st.infeasible and len(fs.queue) == st.added, st
    kids = fs.queue.pick(len(fs.queue), float('inf'))
    for i in range(kids.B):
        side = 0 if float(kids.ub[dec[0] + 1][i, dec[1]]) == 0.0 else 1
        ol, ou, _ = KW.child_bounds(net, x, eps, wp, bp, lbs, ubs, dec, side)
        for k in range(net.L + 2):
            e = max(_err(kids.lb[k][i], ol[k]), _err(kids.ub[k][i], ou[k]))
            assert e <= KW_TOL, (name, 'child', i, k, e)
        assert float(kids.lower_bound[i]) == float(kids.lb[net.L + 1][i, 0])
        assert int(kids.mask[i, sum(net.hidden_sizes[:dec[0]]) + dec[1]]) == side
    fs.queue.add(kids)
    glb, size = fs.queue.global_lb, kids.B
    for B in (2, 4, 8, 16):
        st = fs.step(B)
        size += st.added - st.picked
        assert st.children == 2 * st.picked and st.added <= st.children - st.infeasible and len(fs.queue) == size, (st, size)
        if size:
            assert st.global_lb >= glb - 1e-6, (st.global_lb, glb)
            glb = st.global_lb
    print(f'frontier_step {name}: root decision {dec}, queue {len(fs.queue)} domains, global lb {glb:.4f}', flush=True)


def _chain(L, width=4, seed=0):
    """L linear layers of ``width`` nodes in a row on a flat input (the layer count is all that matters here)."""
    g = torch.Generator().manual_seed(seed)
    layers = [Flatten()]
    for _ in range(L):
        layers += _lin(width, width)
    for m in layers:
        for q in m.parameters():
            q.requires_grad = False
            q.data = torch.randn(q.shape, generator=g) * (0.6 if q.dim() > 1 else 0.1)
    net = netspec_from_modules(layers, (1, 1, width), name=f'chain{L}')
    return net, torch.randn(width, generator=g), torch.randn(width, generator=g) * 0.3


def check_limits(_):
    """Past each size limit the entry point returns GNNB_ERR_UNSUPPORTED (before launching anything) and the context keeps
    working: 16 hidden layers in the domain queue, 17 refused; 30 in the KW bounds, 31 refused; 32 in BaBSR, 33 refused; conv
    weights of exactly 64 KB accepted and scored, 4 bytes per tap more refused with the previous network left in place.
    After every refusal the same context scores base against the reference's committed scores."""
    from gnn_branching_b200 import DomainQueue, Frontier, Scorer, _lib
    from golden_io import load_case
    from oracle import babsr_oracle as BO
    from test_gpu_parity import _check_payload, _queue_batch
    fr_base, ref = load_case('base', 'fr')
    sc = Scorer(0, math='tc')
    sc.set_gnn(load_gnn('random'))

    def base_ok(what, set_net=True):
        if set_net:
            sc.set_network(fr_base.net, key=fr_base.net.key)
        _, idx, scores = sc.score(fr_base.to('cuda'))
        rep = O.parity_report(scores.cpu(), ref['scores_random'], fr_base.mask, idx.cpu(), rtol=RTOL['tc'])
        assert rep['ok'], (what, rep)

    def refused(call, what):
        try:
            call()
        except _lib.GnnbError as e:
            assert e.status == _lib.GNNB_ERR_UNSUPPORTED, (what, str(e))
            return
        raise AssertionError(f'{what}: not refused')

    base_ok('start')
    # domain queue: the row-copy table holds 2 (L + 2) arrays
    for L in (QUEUE_MAX_LAYERS, QUEUE_MAX_LAYERS + 1):
        net = _chain(L)[0]
        sc.set_network(net, key=net.key)
        if L <= QUEUE_MAX_LAYERS:
            q = DomainQueue(sc, capacity=8)
            assert q.add(_queue_batch(net, [0.5, -1.0, 0.25], [3, 1, 2])) == 3
            b = q.pick(3, float('inf'))                   # lowest lower bound first
            _check_payload(net, b, [1, 2, 3])
            del q, b
        else:
            refused(lambda: DomainQueue(sc, capacity=8), f'queue L={L}')
            base_ok(f'queue L={L}')
    # KW bounds: pointer tables of KW_MAX_LAYERS + 1 arrays
    for L in (KW_MAX_LAYERS, KW_MAX_LAYERS + 1):
        net, x, wp = _chain(L, seed=1)
        sc.set_network(net, key=net.key)
        args = (x.reshape(1, -1), 0.05, wp.reshape(1, -1), torch.tensor([0.1]))
        if L <= KW_MAX_LAYERS:
            gl, gu = sc.kw_bounds(*args)
            _check_bounds(gl, gu, 0, *KW.kw_bounds(net, x, 0.05, wp, 0.1), f'kw_bounds L={L}')
        else:
            refused(lambda: sc.kw_bounds(*args), f'kw_bounds L={L}')
            refused(lambda: sc.root_bounds(*args), f'root_bounds L={L}')
            sizes = [net.n0] + net.hidden_sizes + [1]
            pl = [torch.full((1, n), -1.0) for n in sizes]
            pu = [torch.full((1, n), 1.0) for n in sizes]
            one = torch.zeros(1, dtype=torch.int32)
            refused(lambda: sc.child_bounds(*args, pl, pu, one, one, one), f'child_bounds L={L}')
            base_ok(f'kw L={L}')
    # BaBSR: per-layer reductions in MAXL shared slots
    for L in (BABSR_MAX_LAYERS, BABSR_MAX_LAYERS + 1):
        net, x, wp = _chain(L, seed=2)
        sc.set_network(net, key=net.key)
        sizes = [net.n0] + net.hidden_sizes + [1]
        g = torch.Generator().manual_seed(L)
        lb = [-torch.rand(4, n, generator=g) - 0.01 for n in sizes]
        ub = [torch.rand(4, n, generator=g) + 0.01 for n in sizes]
        e = torch.empty(0)
        fr = Frontier(net=net, lb=lb, ub=ub, dual=[], prim_pre=[], prim_post=[], prim_out=e, primal_input=e,
                      Wp=wp.reshape(1, -1).repeat(4, 1), bp=torch.full((4,), 0.1), mask=torch.ones(4, net.n_hidden))
        if L <= BABSR_MAX_LAYERS:
            dec, cout, kind, scores = sc.babsr(fr.to('cuda'), None, list(range(L)), 0, 0.001, return_scores=True)
            s_or, ic = BO.babsr_scores(fr)
            assert float((scores.cpu() - s_or).abs().max()) <= BABSR_RTOL * float(s_or.abs().max()), f'babsr L={L}'
        else:
            refused(lambda: sc.babsr(fr.to('cuda'), None, list(range(L)), 0, 0.001), f'babsr L={L}')
            base_ok(f'babsr L={L}')
    # conv weights: staged in a 64 KB shared-memory buffer
    def conv_net(co):
        layers = _conv(4, co, 4, 1, 0) + [Flatten()] + _lin(co, 3)
        g = torch.Generator().manual_seed(co)
        for m in layers:
            for q in m.parameters():
                q.requires_grad = False
                q.data = torch.randn(q.shape, generator=g) * (0.3 if q.dim() > 1 else 0.1)
        return netspec_from_modules(layers, (4, 4, 4), name=f'conv{co}'), torch.randn(64, generator=g)
    net, x = conv_net(256)
    assert 4 * 256 * 4 * 4 * 4 == CONV_WEIGHT_MAX_BYTES
    sc.set_network(net, key=net.key)
    wp = torch.randn(net.hidden_sizes[-1], generator=torch.Generator().manual_seed(5)) * 0.3
    lbs, ubs = KW.root_bounds(net, x, 0.05, wp, 0.1)
    fr = synthetic_frontier(net, lbs, ubs, wp, 0.1, 16, seed=5, max_splits=4)
    _, idx, scores = sc.score(fr.to('cuda'))
    s_or, _ = O.gnn_forward(load_gnn('random'), fr)
    rep = O.parity_report(scores.cpu(), s_or, fr.mask, idx.cpu(), rtol=RTOL['tc'])
    assert rep['ok'], ('64 KB conv weights', rep)
    base_ok('before the conv refusal')
    big = conv_net(257)[0]
    refused(lambda: sc.set_network(big, key=big.key), 'conv weights of 64 KB + 64 bytes')
    assert sc.net is fr_base.net
    base_ok('conv weights refused', set_net=False)
    print('limits: every refusal returned GNNB_ERR_UNSUPPORTED and left the context usable', flush=True)


if __name__ == '__main__':
    {'kw': check_kw, 'frontier_step': check_frontier_step, 'limits': check_limits}[sys.argv[1]](sys.argv[2])
    print('ok')
