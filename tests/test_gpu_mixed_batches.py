"""The batched entry points on frontiers whose subdomains differ in input point and property.

Every batched call takes per-subdomain rows: ``wp [B, n_L]``, ``bp [B]`` of the folded property layer and, for the KW bounds,
``x [B, n0]``.  A frontier here mixes K roots, each with its own (x, wp, bp) and its own KW root bounds, and interleaves their
subdomains with a fixed permutation, so neighbouring subdomains, waves, CTA groups and the second KW pass's domain list all
mix properties.  A kernel that read such a row at the wrong subdomain (domain 0's row, the wave-local or the list-local
row) gives a wrong answer here; every comparison first checks that the oracle under property 0 is far from the oracle under
the subdomain's own property, so that such a bug cannot pass.

Scoring, BaBSR and gradients run in the pytest process; the KW bound checks run in their own process (`_run_isolated`:
python tests/test_gpu_mixed_batches.py <check> <arg>, exit code 0 = pass).
"""
import functools
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import ctypes as C                                               # noqa: E402

import numpy as np                                               # noqa: E402
import pytest                                                    # noqa: E402
import torch                                                     # noqa: E402

from golden_io import GOLDEN, load_gnn, load_root                # noqa: E402
from gnn_branching_b200 import Frontier, GraphNet, Scorer, synthetic_frontier, _lib      # noqa: E402
from oracle import graphnet_oracle as O                          # noqa: E402
from oracle import kw_bounds_oracle as KW                        # noqa: E402

pytestmark = pytest.mark.gpu

RTOL = {'simt': 1e-5, 'tc': 1e-4}
KW_TOL = 5e-5                   # KW bounds: max|got - want| <= KW_TOL * max(1, max|want|) per layer
GUARD = 100                     # the oracle under property 0 must be this many tolerances away from the right answer
SCORE_B = {'base': 1000, 'deep': 1000, 'odd_shapes': 300, 'wide_channels': 300}


# ---- networks and roots ------------------------------------------------------------------------------------------------
def _custom_net(case):
    """(net, x, wp, bp, eps).  odd_shapes / wide_channels: the nets of test_gpu_parity._custom_frontier (odd spatial sizes and
    channel counts, > 128 channels); tiny: conv -> conv -> linear, small enough for frontiers past 65 535 domains."""
    from torch import nn
    from gnn_branching_b200 import Flatten, netspec_from_modules
    if case == 'odd_shapes':
        layers = [nn.Conv2d(2, 5, 3, stride=1, padding=1), nn.ReLU(), nn.Conv2d(5, 6, 3, stride=2, padding=1), nn.ReLU(),
                  Flatten(), nn.Linear(6 * 5 * 4, 37), nn.ReLU()]
        shape = (2, 9, 7)
    elif case == 'wide_channels':
        layers = [nn.Conv2d(3, 130, 3, stride=1, padding=1), nn.ReLU(), Flatten(), nn.Linear(130 * 4 * 4, 20), nn.ReLU()]
        shape = (3, 4, 4)
    else:
        layers = [nn.Conv2d(1, 8, 3, stride=1, padding=1), nn.ReLU(), nn.Conv2d(8, 8, 4, stride=2, padding=1), nn.ReLU(),
                  Flatten(), nn.Linear(8 * 4 * 4, 10), nn.ReLU()]
        shape = (1, 8, 8)
    g = torch.Generator().manual_seed(11)
    for m in layers:
        for q in m.parameters():
            q.data = torch.randn(q.shape, generator=g) * (0.3 if q.dim() > 1 else 0.1)
    net = netspec_from_modules(layers, shape, name=case)
    x = torch.randn(shape, generator=g).reshape(-1)
    wp = torch.randn(net.hidden_sizes[-1], generator=g) * 0.3
    return net, x, wp, 0.1, 0.05


def _base_root(name):
    if name in ('base', 'wide', 'deep'):
        net, _, _, wp, bp = load_root(name)
        x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))[f'{name}_x'].copy()).reshape(-1)
        return net, x, wp, bp, 0.145
    return _custom_net(name)


@functools.lru_cache(maxsize=None)
def _roots(name, K, eps=None):
    """(net, eps, roots): root 0 is the net's own (x, wp, bp); odd roots keep x and take another property (wp permuted,
    sign-flipped and rescaled, another bp), even roots take another point too (x plus clipped noise).  Every root carries its
    KW root bounds (oracle)."""
    net, x, wp, bp, eps0 = _base_root(name)
    eps = eps0 if eps is None else eps
    g = torch.Generator().manual_seed(1000 + K)
    lo, hi = float(x.min()), float(x.max())
    roots = []
    for r in range(K):
        xr, wr, br = x, wp, float(bp)
        if r > 0:
            n = wp.numel()
            sign = torch.where(torch.rand(n, generator=g) < 0.5, -1.0, 1.0)
            wr = wp[torch.randperm(n, generator=g)] * sign * (0.6 + 0.8 * float(torch.rand(1, generator=g)))
            br = float(bp) + 0.5 * float(torch.randn(1, generator=g))
        if r > 0 and r % 2 == 0:
            xr = (x + (0.05 * torch.randn(x.shape, generator=g)).clamp(-0.1, 0.1)).clamp(lo, hi)
        lbs, ubs = KW.root_bounds(net, xr, eps, wr, br)
        # parent bounds for child domains: the root's, with a property output bound 10 looser, so that a child's output bound
        # is its own KW bound (which depends on its x, wp, bp) and not the parent's
        plb, pub = lbs[:-1] + [lbs[-1] - 10], ubs[:-1] + [ubs[-1] + 10]
        roots.append(dict(x=xr, wp=wr, bp=br, lbs=lbs, ubs=ubs, plb=plb, pub=pub))
    return net, eps, roots


def _cat(frs):
    out = {}
    for k, v in frs[0].tensors().items():
        if isinstance(v, list):
            out[k] = [torch.cat([f.tensors()[k][i] for f in frs]) for i in range(len(v))]
        else:
            out[k] = torch.cat([f.tensors()[k] for f in frs])
    return Frontier(net=frs[0].net, **out)


@functools.lru_cache(maxsize=None)
def _mixed(name, B, K=4, seed=7):
    """(frontier on the CPU, root of every subdomain [B]): synthetic_frontier of every root, concatenated, interleaved."""
    net, _, roots = _roots(name, K)
    sizes = [B // K + (r < B % K) for r in range(K)]
    splits = 32 if name in ('base', 'wide', 'deep') else 4
    parts = [synthetic_frontier(net, r['lbs'], r['ubs'], r['wp'], r['bp'], n, seed=seed + 100 * i, max_splits=splits)
             for i, (r, n) in enumerate(zip(roots, sizes))]
    root = torch.cat([torch.full((n,), i, dtype=torch.long) for i, n in enumerate(sizes)])
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(seed))
    return _cat(parts)._map(lambda t: t[perm].contiguous()), root[perm]


def _with_property(fr, wp, bp):
    """``fr`` with every subdomain's property replaced by (wp, bp)."""
    out = fr._map(lambda t: t)
    out.Wp = wp.reshape(1, -1).expand(fr.B, -1).contiguous()
    out.bp = torch.full((fr.B,), float(bp))
    return out


def _bits(t):
    return t.contiguous().view(torch.int32)


def _spread(B, root, K):
    """About 16 subdomains spread over the batch (first and last waves, around the middle, the tail) and at least one of
    every root."""
    ids = {0, 1, 6, 7, 8, B // 5, B // 3, B // 2 - 1, B // 2, (2 * B) // 3, B - 130, B - 9, B - 8, B - 3, B - 2, B - 1}
    for r in range(K):
        ids.add(int((root == r).nonzero()[0]))
    ids = sorted(i for i in ids if 0 <= i < B)
    assert set(root[ids].tolist()) == set(range(K))
    return ids


def _row_err(a, b, mask):
    """max over candidates |a - b| / max |b| per row."""
    m = mask != 0
    d = torch.where(m, (a - b).abs(), torch.zeros_like(a)).amax(1)
    s = torch.where(m, b.abs(), torch.zeros_like(b)).amax(1)
    return d / s.clamp(min=1e-30)


# ---- scoring ------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _score_case(name):
    """The mixed frontier, the oracle's scores of a spread of its subdomains, and the guard: under root 0's property the
    oracle's scores of the other roots' subdomains move by far more than the tolerance."""
    B = SCORE_B[name]
    net, _, roots = _roots(name, 4)
    fr, root = _mixed(name, B)
    ids = _spread(B, root, 4)
    sl = fr._map(lambda t: t[ids].contiguous())
    sd = load_gnn('random')
    s_or, _ = O.gnn_forward(sd, sl)
    s_p0, _ = O.gnn_forward(sd, _with_property(sl, roots[0]['wp'], roots[0]['bp']))
    other = root[ids] != 0
    moved = _row_err(s_p0, s_or, sl.mask)[other]
    assert float(moved.min()) > GUARD * RTOL['tc'], (name, moved)
    return dict(fr=fr, root=root, ids=ids, s_or=s_or, net=net, roots=roots)


def _scorer(net, math, chunk=0, fuse=1, rescore=False):
    model = GraphNet(2, 64, math=math, chunk=chunk, rescore=rescore)
    model.load_state_dict(load_gnn('random'))
    sc = model.eval().cuda().scorer(0)
    sc.set_network(net, key=net.key)
    if math == 'tc':
        sc.set_option('fuse', fuse)
    return sc


def _score(sc, fr, mem):
    best, idx, scores = sc.score(fr.to('cuda') if mem == 'device' else fr.pin())
    torch.cuda.synchronize()
    return best.cuda(), idx.cuda(), scores.cuda()


def _same(a, b):
    return all(torch.equal(_bits(x) if x.dtype == torch.float32 else x, _bits(y) if y.dtype == torch.float32 else y) for x, y in zip(a, b))


@pytest.mark.parametrize('math', ['tc', 'simt'])
@pytest.mark.parametrize('name', list(SCORE_B))
def test_scores_follow_their_own_property(name, math):
    """Per fuse mode: oracle parity on the spread; chunk 7 (waves of 7 that cut through every CTA group) and pinned host buffers
    give bit-identical results; scoring F[perm] gives outputs[perm] bit for bit; winner records and top-k column 0 are the
    scores' winners and the top-k is gnnb_topk of the dense scores; changing one subdomain's wp / bp changes its scores and no
    other subdomain's."""
    c = _score_case(name)
    fr, root, ids = c['fr'], c['root'], c['ids']
    B = fr.B
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(3))
    for fuse in ([1, 0] if math == 'tc' else [1]):
        sc0, sc7 = _scorer(c['net'], math, 0, fuse), _scorer(c['net'], math, 7, fuse)
        ref = _score(sc0, fr, 'device')
        best, idx, scores = ref
        rep = O.parity_report(scores[ids].cpu(), c['s_or'], fr.mask[ids], idx[ids].cpu(), rtol=RTOL[math])
        assert rep['ok'], (fuse, rep)
        m = fr.mask.cuda() != 0
        assert torch.equal(torch.where(m, scores, torch.full_like(scores, float('-inf'))).max(1).values, best)
        assert _same(_score(sc7, fr, 'host'), ref), ('chunk 7, host buffers', fuse)
        assert _same(_score(sc7, fr, 'device'), ref), ('chunk 7, device buffers', fuse)
        fp = fr._map(lambda t: t[perm].contiguous())
        for sc, mem in ((sc0, 'device'), (sc7, 'host')):
            assert _same(_score(sc, fp, mem), [t[perm.cuda()] for t in ref]), ('permuted frontier', fuse, mem)
        # winner records and top-k
        fd = fr.to('cuda')
        rec = sc7.score_winners(fd)
        torch.cuda.synchronize()
        assert torch.equal(rec[:, 0], _bits(best)) and torch.equal(rec[:, 1], idx)
        ts, ti, s2 = sc7.score_topk(fd, 5, return_scores=True)
        assert torch.equal(_bits(s2), _bits(scores))
        assert torch.equal(_bits(ts[:, 0]), _bits(best)) and torch.equal(ti[:, 0], idx)
        rs, ri = sc0.topk(scores, 5, fd.mask)
        assert torch.equal(_bits(ts), _bits(rs)) and torch.equal(ti, ri)
        # one subdomain takes another root's property: its row changes by far more than the tolerance, no other row changes
        j = ids[len(ids) // 2]
        other = (int(root[j]) + 1) % 4
        f1 = fr._map(lambda t: t.clone())
        f1.Wp[j] = c['roots'][other]['wp']
        f1.bp[j] = c['roots'][other]['bp']
        b1, i1, s1 = _score(sc7, f1, 'device')
        keep = torch.arange(B, device='cuda') != j
        assert _same((b1[keep], i1[keep], s1[keep]), (best[keep], idx[keep], scores[keep])), ('other rows moved', fuse)
        moved = float(_row_err(s1[j:j + 1].cpu(), scores[j:j + 1].cpu(), fr.mask[j:j + 1]))
        assert moved > GUARD * RTOL[math], ('row did not follow its property', fuse, moved)


FACTORS = [1e6, 1e7, 1e8, 1e9, 1e10]


def _nan_status(sc):
    """Status of gnnb_check: the sticky NaN report of the last device call."""
    n = C.c_int64(0)
    return sc.lib.gnnb_check(sc.h, C.c_void_p(torch.cuda.current_stream().cuda_stream), C.byref(n))


@pytest.mark.parametrize('fuse', [1, 0])
def test_rescore_gathers_the_rows_of_their_own_property(fuse):
    """Option rescore on the mixed base frontier: four subdomains of four roots overflow the tensor-core range (duals scaled);
    they are scored again in exact fp32 from gathered rows (k_gather_rows on device buffers, row copies on pinned host
    buffers, chunk 7) and equal the SIMT mode's rows bit for bit; every other row keeps its tensor-core result bit for bit."""
    c = _score_case('base')
    fr0, root = c['fr'], c['root']
    rows = [int((root == r).nonzero()[3 + 5 * r]) for r in range(4)]
    tc, simt = _scorer(c['net'], 'tc', fuse=fuse), _scorer(c['net'], 'simt')
    for f in FACTORS:
        fr = fr0._map(lambda t: t.clone())
        for d in fr.dual:
            d[rows] *= f
        sc_off = tc.score(fr.to('cuda'), check=False)
        torch.cuda.synchronize()
        if _nan_status(tc) != _lib.GNNB_ERR_NAN:
            continue
        ref = _score(simt, fr, 'device')
        if _nan_status(simt) != _lib.GNNB_OK or not bool(torch.isfinite(ref[2][rows]).all()):
            continue
        break
    else:
        pytest.fail(f'no factor in {FACTORS} overflows the tensor-core path with a finite fp32 result')
    keep = torch.ones(fr.B, dtype=torch.bool, device='cuda')
    keep[rows] = False
    for chunk, mem in ((0, 'device'), (7, 'host')):
        sc = _scorer(c['net'], 'tc', chunk, fuse, rescore=True)
        got = _score(sc, fr, mem)
        assert sc.rescored == len(rows), (chunk, mem, sc.rescored)
        assert _same([t[rows] for t in got], [t[rows] for t in ref]), ('re-scored rows', chunk, mem)
        assert _same([t[keep] for t in got], [t[keep] for t in sc_off]), ('other rows', chunk, mem)


# ---- BaBSR -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('mem', ['device', 'host'])
@pytest.mark.parametrize('arch', ['base', 'deep'])
def test_babsr_follows_its_own_property(arch, mem):
    """gnnb_babsr on the mixed frontier: scores within 1e-5 of the largest oracle score, decisions and counters equal to the
    oracle's wherever its top-2 margin is safe; the oracle's scores under root 0's property are far from them."""
    from oracle import babsr_oracle as BO
    c = _score_case(arch)
    fr, root, net = c['fr'], c['root'], c['net']
    order = [0] + [k for k in range(net.L) if k != 0]
    sc = Scorer(0)
    sc.set_network(net, key=net.key)
    dec, cout, kind, scores = sc.babsr(fr.to('cuda') if mem == 'device' else fr, None, order, 0, 0.001, return_scores=True)
    torch.cuda.synchronize()
    s_or, ic = BO.babsr_scores(fr)
    tol = 1e-5 * float(s_or.abs().max())
    assert float((scores.cpu() - s_or).abs().max()) <= tol
    s_p0, _ = BO.babsr_scores(_with_property(fr, c['roots'][0]['wp'], c['roots'][0]['bp']))
    other = root != 0
    assert float((s_p0 - s_or).abs().amax(1)[other].min()) > GUARD * tol
    d_or, c_or, _ = BO.babsr_decide(s_or, ic, fr.mask, net.hidden_sizes, [0] * fr.B, order, 0, 0.001)
    top2 = s_or.topk(2, dim=1).values
    safe = (top2[:, 0] - top2[:, 1]) > 2 * tol
    assert int(safe.sum()) > fr.B // 2
    assert torch.equal(dec.cpu()[safe].long(), d_or[safe]) and torch.equal(cout.cpu()[safe].long(), c_or[safe])


# ---- gradients ---------------------------------------------------------------------------------------------------------
def _grad_frontier(name, B):
    """B subdomains of the mixed frontier, one of each of the first B roots."""
    c = _score_case(name)
    pick = [int((c['root'] == r).nonzero()[0]) for r in range(B)]
    return c['fr']._map(lambda t: t[pick].contiguous()), c['net']


def _terms(fr):
    terms = []
    for b in range(fr.B):
        cand = fr.mask[b].nonzero().view(-1).tolist()
        terms += [(b, cand[0], 1.0), (b, cand[len(cand) // 2], -0.5 - b), (b, cand[-1], 0.25)]
    return terms


@pytest.mark.parametrize('name,B', [('base', 4), ('odd_shapes', 3)])
def test_score_grad_is_the_sum_of_single_domain_gradients(name, B):
    """gnnb_score_grad is batch invariant in its forward (term scores equal single-domain calls bit for bit), so the batched
    gradient is the sum of the single-domain gradients up to the order of the atomicAdds (1e-5 of sum_b max|g_b| per tensor);
    two terms on one (domain, index) with coefficients a and c give the gradient of one term with a + c."""
    fr, net = _grad_frontier(name, B)
    sc = _scorer(net, 'tc')
    fd = fr.to('cuda')
    terms = _terms(fr)
    vals = sc.score_grad(fd, terms)
    g = sc.gradients()
    singles, single_vals = [], []
    for b in range(B):
        mine = [(0, i, cf) for d, i, cf in terms if d == b]
        single_vals.append(sc.score_grad(fd.slice(b, b + 1).contiguous(), mine))
        singles.append(sc.gradients())
    assert torch.equal(_bits(vals), _bits(torch.cat(single_vals))), 'the batched forward is not batch invariant'
    tol = {k: 1e-5 * sum(float(s[k].abs().max()) for s in singles) for k in g}
    for k in g:
        err = float((g[k] - sum(s[k] for s in singles)).abs().max())
        assert err <= tol[k], (k, err, tol[k])
    assert max(float(g[k].abs().max()) for k in g) > 0
    # the first term of domain 1 split in two
    d, i, cf = terms[3]
    split = terms[:3] + [(d, i, 0.75 * cf), (d, i, 0.25 * cf)] + terms[4:]
    vals2 = sc.score_grad(fd, split)
    assert torch.equal(_bits(vals2[3]), _bits(vals[3])) and torch.equal(_bits(vals2[4]), _bits(vals[3]))
    g2 = sc.gradients()
    for k in g:
        err = float((g2[k] - g[k]).abs().max())
        assert err <= tol[k], ('split term', k, err, tol[k])


def test_score_grad_other_network_shapes_match_oracle():
    """odd_shapes (stride 1 and 2, 3x3 kernels on 9x7 and 5x4 maps, clipped windows) against the autograd oracle at the batched
    tolerance of test_gpu_parity (ReLU masks may flip between two fp32 evaluations)."""
    from oracle import online_oracle as OO
    from test_gpu_parity import _assert_grads
    fr, net = _grad_frontier('odd_shapes', 3)
    terms = _terms(fr)
    ref, vals_ref = OO.score_grads(load_gnn('random'), fr, terms)
    sc = _scorer(net, 'tc')
    for dev in ('cuda', 'cpu'):
        vals = sc.score_grad(fr.to(dev), terms)
        assert float((vals - vals_ref).abs().max()) <= 1e-5 * float(vals_ref.abs().max())
        _assert_grads(sc.gradients(), ref, rtol=2e-2)


# ---- KW bounds (own process) -------------------------------------------------------------------------------------------
def _iso(what, arg, timeout=240, math='0'):
    from test_gpu_parity import _run_isolated
    _run_isolated(what, arg, timeout=timeout, env={'GNNB_TEST_MATH': math}, script=os.path.basename(__file__))


@pytest.mark.parametrize('math', ['0', '1'])
@pytest.mark.parametrize('arch', ['base', 'wide', 'deep'])
def test_kw_bounds_per_domain_rows(arch, math):
    _iso('kw_bounds', arch, math=math)


@pytest.mark.parametrize('math', ['0', '1'])
@pytest.mark.parametrize('arch', ['base', 'deep'])
def test_root_bounds_of_several_roots(arch, math):
    _iso('root_bounds', arch, math=math)


@pytest.mark.parametrize('math', ['0', '1'])
@pytest.mark.parametrize('case', ['base', 'odd_shapes'])
def test_child_bounds_second_pass_on_a_domain_list(case, math):
    _iso('child_bounds', case, math=math)


@pytest.mark.parametrize('math', ['0', '1'])
def test_child_bounds_past_the_cone_grid_limit(math):
    _iso('cone_grid', 'tiny', timeout=400, math=math)


def test_child_bounds_on_two_devices():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two visible GPUs')
    _iso('two_devices', 'wide')


def _kw_scorer(net):
    sc = Scorer(0)
    sc.set_network(net, key=net.key)
    sc.set_option('math', int(os.environ.get('GNNB_TEST_MATH', '0')))      # 0: dense layers on the tensor cores, 1: exact fp32
    return sc


def _err(a, b):
    return float((a.reshape(-1).cpu() - b.reshape(-1)).abs().max()) / max(1.0, float(b.abs().max()))


def _check_bounds(gl, gu, i, want_l, want_u, what):
    worst = 0.0
    for k in range(len(want_l)):
        e = max(_err(gl[k][i], want_l[k]), _err(gu[k][i], want_u[k]))
        worst = max(worst, e)
        assert e <= KW_TOL, (what, i, k, e)
    return worst


def _guard(own, p0, what):
    """The property output's bounds under root 0's (x, wp, bp) are far from the domain's own."""
    e = max(_err(p0[0][-1], own[0][-1]), _err(p0[1][-1], own[1][-1]))
    assert e > GUARD * KW_TOL, (what, 'vacuous: root 0 gives nearly the same bounds', e)


def _order(K, B, seed):
    """Root of every domain: each root at least once, in a fixed shuffled order."""
    g = torch.Generator().manual_seed(seed)
    r = torch.cat([torch.arange(K), torch.randint(0, K, (B - K,), generator=g)])
    return r[torch.randperm(B, generator=g)]


def check_kw_bounds(arch):
    """gnnb_kw_bounds with per-domain x, wp, bp (12 domains of 6 roots) against KW.kw_bounds domain by domain."""
    net, eps, roots = _roots(arch, 6)
    r = _order(6, 12, 1)
    X = torch.stack([roots[i]['x'] for i in r.tolist()])
    WP = torch.stack([roots[i]['wp'] for i in r.tolist()])
    BP = torch.tensor([roots[i]['bp'] for i in r.tolist()])
    sc = _kw_scorer(net)
    gl, gu = sc.kw_bounds(X, eps, WP, BP)
    want = [KW.kw_bounds(net, q['x'], eps, q['wp'], q['bp']) for q in roots]
    worst = 0.0
    for i, ri in enumerate(r.tolist()):
        worst = max(worst, _check_bounds(gl, gu, i, *want[ri], 'kw_bounds'))
        if ri:
            _guard(want[ri], want[0], ('kw_bounds', i))
    print(f'kw_bounds {arch} math={sc.get_option("math")}: 12 domains of 6 roots, worst rel err {worst:.2e}', flush=True)


def _root_moved(net, x, eps, wp, bp):
    """How far the interval bounds move the KW root bounds of a hidden layer (the reference's test: a second KW pass above
    1e-4); the same steps as KW.root_bounds."""
    k_lbs, k_ubs = KW.kw_bounds(net, x, eps, wp, bp)
    lbs, ubs, moved = [k_lbs[0]], [k_ubs[0]], 0.0
    for k in range(1, net.L + 1):
        lo_post, hi_post = (lbs[k - 1], ubs[k - 1]) if k == 1 else (lbs[k - 1].clamp(min=0), ubs[k - 1].clamp(min=0))
        lo, hi = KW.interval_layer(net.affine[k - 1], lo_post, hi_post)
        lbs.append(torch.max(k_lbs[k], lo))
        ubs.append(torch.min(k_ubs[k], hi))
        moved = max(moved, float((lbs[k] - k_lbs[k]).abs().max()), float((ubs[k] - k_ubs[k]).abs().max()))
    return moved


def check_root_bounds(arch):
    """gnnb_root_bounds on 8 roots of 6 (x, wp, bp): bounds against KW.root_bounds, the BaB masks from the bounds, the
    second-pass flags against the oracle's "a hidden layer moved by more than 1e-4" wherever that is not within rounding."""
    net, eps, roots = _roots(arch, 6)
    r = _order(6, 8, 2)
    X = torch.stack([roots[i]['x'] for i in r.tolist()])
    WP = torch.stack([roots[i]['wp'] for i in r.tolist()])
    BP = torch.tensor([roots[i]['bp'] for i in r.tolist()])
    sc = _kw_scorer(net)
    gl, gu, masks, second = sc.root_bounds(X, eps, WP, BP)
    torch.cuda.synchronize()
    moved = [_root_moved(net, q['x'], eps, q['wp'], q['bp']) for q in roots]
    worst = 0.0
    for i, ri in enumerate(r.tolist()):
        q = roots[ri]
        worst = max(worst, _check_bounds(gl, gu, i, q['lbs'], q['ubs'], 'root_bounds'))
        if ri:
            _guard((q['lbs'], q['ubs']), (roots[0]['lbs'], roots[0]['ubs']), ('root_bounds', i))
        for k in range(1, net.L + 1):
            l, u = gl[k][i].cpu(), gu[k][i].cpu()
            want = torch.where((l >= 0) & (u >= 0), 1, torch.where((l <= 0) & (u <= 0), 0, -1)).to(torch.int8)
            assert torch.equal(masks[k - 1][i].cpu(), want), ('mask', i, k)
        if not 0.5e-4 < moved[ri] < 2e-4:
            assert int(second[i]) == int(moved[ri] > 1e-4), ('second pass', i, int(second[i]), moved[ri])
    print(f'root_bounds {arch} math={sc.get_option("math")}: 8 roots, second passes {second.tolist()}, moved '
          f'{[f"{m:.1e}" for m in moved]}, worst rel err {worst:.2e}', flush=True)


def _decisions(net, roots, r, want_second, g):
    """A split per domain on an ambiguous ReLU of its root: in the last hidden layer (nothing behind it, never a second pass)
    where want_second is 0, in front of it where the oracle takes the second pass otherwise (or, when 64 tries find no such
    split of that root, in the last layer).  Returns the decisions and the oracle's (lbs, ubs) per domain."""
    L = net.L
    out, want = [], []
    for ri, sec in zip(r.tolist(), want_second):
        q = roots[ri]
        for attempt in range(65):
            lay = L - 1 if not sec or attempt == 64 else int(torch.randint(0, L - 1, (1,), generator=g))
            amb = ((q['lbs'][lay + 1] < 0) & (q['ubs'][lay + 1] > 0)).nonzero().view(-1)
            if amb.numel() == 0:
                continue
            dec = (lay, int(amb[int(torch.randint(0, amb.numel(), (1,), generator=g))]), int(torch.randint(0, 2, (1,), generator=g)))
            ol, ou, changed = KW.child_bounds(net, q['x'], q['eps'], q['wp'], q['bp'], q['plb'], q['pub'], dec[:2], dec[2])
            if bool(changed) == bool(sec) or lay == L - 1:
                break
        else:
            raise AssertionError(f'root {ri} has no ambiguous ReLU in its last hidden layer')
        out.append(dec)
        want.append((ol, ou))
    return out, want


def _child_call(sc, net, eps, roots, r, decs, rows=None):
    rows = list(range(len(decs))) if rows is None else rows
    rr = [r[i] for i in rows]
    X = torch.stack([roots[i]['x'] for i in rr])
    WP = torch.stack([roots[i]['wp'] for i in rr])
    BP = torch.tensor([roots[i]['bp'] for i in rr])
    plb = [torch.stack([roots[i]['plb'][k] for i in rr]) for k in range(net.L + 2)]
    pub = [torch.stack([roots[i]['pub'][k] for i in rr]) for k in range(net.L + 2)]
    dec = torch.tensor([decs[i] for i in rows], dtype=torch.int32).reshape(-1, 3)
    out = sc.child_bounds(X, eps, WP, BP, plb, pub, dec[:, 0], dec[:, 1], dec[:, 2])
    torch.cuda.synchronize()
    return out


def check_child_bounds(case):
    """gnnb_child_bounds on 12 children of parents from 6 roots (each its own x, wp, bp and KW root bounds) whose second KW pass
    runs on a proper, non-contiguous subset (dom_list is neither all domains nor a prefix): bounds against KW.child_bounds, the
    flags of the last-layer splits 0, and the permuted batch gives the permuted results bit for bit.  base: the cone kernel's
    vector path (16 channels), odd_shapes: its scalar path (6 channels), at eps = 0.5 (at 0.05 no split of this net takes the
    second pass)."""
    net, eps, roots = _roots(case, 6, 0.5 if case == 'odd_shapes' else None)
    for q in roots:
        q['eps'] = eps
    B = 12
    r = _order(6, B, 3)
    want_second = [1 if i % 3 == 1 else 0 for i in range(B)]
    g = torch.Generator().manual_seed(4)
    decs, want = _decisions(net, roots, r, want_second, g)
    sc = _kw_scorer(net)
    r_list = r.tolist()
    gl, gu, masks, second = _child_call(sc, net, eps, roots, r_list, decs)
    sec = second.cpu()
    n2 = int(sec.sum())
    assert 0 < n2 < B and not bool(sec[:n2].all()), ('the second pass does not run on a proper non-prefix subset', sec.tolist())
    worst = 0.0
    for i in range(B):
        worst = max(worst, _check_bounds(gl, gu, i, *want[i], 'child_bounds'))
        if decs[i][0] == net.L - 1:
            assert int(sec[i]) == 0, ('second pass behind the last hidden layer', i)
        if r_list[i]:
            q = roots[0]
            p0 = KW.child_bounds(net, q['x'], eps, q['wp'], q['bp'], roots[r_list[i]]['plb'], roots[r_list[i]]['pub'], decs[i][:2], decs[i][2])
            _guard(want[i], p0, ('child_bounds', i))
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(5)).tolist()
    pl, pu, pm, ps = _child_call(sc, net, eps, roots, r_list, decs, rows=perm)
    for k in range(net.L + 2):
        assert torch.equal(_bits(pl[k]), _bits(gl[k][perm])) and torch.equal(_bits(pu[k]), _bits(gu[k][perm])), ('permuted', k)
    for k in range(net.L):
        assert torch.equal(pm[k], masks[k][perm])
    assert torch.equal(ps, second[perm])
    print(f'child_bounds {case} math={sc.get_option("math")}: {B} children, second pass on {sec.nonzero().view(-1).tolist()}, '
          f'worst rel err {worst:.2e}', flush=True)


def check_cone_grid(case):
    """gnnb_child_bounds on 65 535 + 300 children of the tiny conv -> conv -> linear net (the cone kernel's grid is split at
    65 535 domains and the later launches shift their per-domain views), per-domain x, wp, bp from 8 roots, and the root of
    every domain past 65 535 differs from the root of the domain 65 535 before it.  Domains 65 530 .. 65 540, the last 3 and 8
    random ones against the oracle; each of them computed alone gives the same bits."""
    net, eps, roots = _roots(case, 8)
    B = 65535 + 300
    g = torch.Generator().manual_seed(6)
    r = torch.randint(0, 8, (B,), generator=g)
    r[65535:] = (r[:300] + 1 + torch.randint(0, 7, (300,), generator=g)) % 8
    L = net.L
    # a random ambiguous ReLU of the domain's root in a random layer
    dec = torch.zeros(B, 3, dtype=torch.int32)
    lay = torch.randint(0, L, (B,), generator=g)
    for ri in range(8):
        for k in range(L):
            amb = ((roots[ri]['lbs'][k + 1] < 0) & (roots[ri]['ubs'][k + 1] > 0)).nonzero().view(-1)
            sel = ((r == ri) & (lay == k)).nonzero().view(-1)
            assert amb.numel() > 0
            dec[sel, 0] = k
            dec[sel, 1] = amb[torch.randint(0, amb.numel(), (sel.numel(),), generator=g)].int()
    dec[:, 2] = torch.randint(0, 2, (B,), generator=g).int()
    X = torch.stack([q['x'] for q in roots])[r]
    WP = torch.stack([q['wp'] for q in roots])[r]
    BP = torch.tensor([q['bp'] for q in roots])[r]
    plb = [torch.stack([q['plb'][k] for q in roots])[r] for k in range(L + 2)]
    pub = [torch.stack([q['pub'][k] for q in roots])[r] for k in range(L + 2)]
    sc = _kw_scorer(net)
    gl, gu, _, second = sc.child_bounds(X, eps, WP, BP, plb, pub, dec[:, 0], dec[:, 1], dec[:, 2], with_mask=False)
    torch.cuda.synchronize()
    check = list(range(65530, 65541)) + [B - 3, B - 2, B - 1] + torch.randint(0, B, (8,), generator=g).tolist()
    worst = 0.0
    for i in check:
        q = roots[int(r[i])]
        d = dec[i].tolist()
        ol, ou, _ = KW.child_bounds(net, q['x'], eps, q['wp'], q['bp'], q['plb'], q['pub'], d[:2], d[2])
        worst = max(worst, _check_bounds(gl, gu, i, ol, ou, 'cone grid'))
        if int(r[i]):
            q0 = roots[0]
            _guard((ol, ou), KW.child_bounds(net, q0['x'], eps, q0['wp'], q0['bp'], q['plb'], q['pub'], d[:2], d[2]), ('cone grid', i))
        al, au, _, _ = sc.child_bounds(X[i:i + 1], eps, WP[i:i + 1], BP[i:i + 1], [t[i:i + 1] for t in plb], [t[i:i + 1] for t in pub],
                                       dec[i:i + 1, 0], dec[i:i + 1, 1], dec[i:i + 1, 2], with_mask=False)
        torch.cuda.synchronize()
        for k in range(L + 2):
            assert torch.equal(_bits(al[k][0]), _bits(gl[k][i])) and torch.equal(_bits(au[k][0]), _bits(gu[k][i])), ('alone', i, k)
    print(f'cone grid {case} math={sc.get_option("math")}: {B} children, {int(second.sum())} second passes, worst rel err '
          f'{worst:.2e}', flush=True)


def check_two_devices(arch):
    """Child bounds on wide (the cone kernel's conv2 launch needs about 77 KB of shared memory, above the 48 KB default) on
    device 0, then on device 1 in the same process: the opt-in is per device, so both succeed, with the same bits."""
    net, eps, roots = _roots(arch, 1)
    q = roots[0]
    amb = ((q['lbs'][2] < 0) & (q['ubs'][2] > 0)).nonzero().view(-1)[:4].tolist()
    decs = [(0, int(((q['lbs'][1] < 0) & (q['ubs'][1] > 0)).nonzero()[0]), 1)] + [(1, i, i % 2) for i in amb]
    outs = []
    for dev in (0, 1):
        sc = Scorer(dev)
        sc.set_network(net, key=net.key)
        with torch.cuda.device(dev):
            gl, gu, _, _ = _child_call(sc, net, eps, [q], [0] * len(decs), decs)
        outs.append([t.cpu() for t in gl + gu])
    for a, b in zip(*outs):
        assert torch.equal(_bits(a), _bits(b))
    print(f'two devices {arch}: {len(decs)} children, identical bounds', flush=True)


if __name__ == '__main__':
    {'kw_bounds': check_kw_bounds, 'root_bounds': check_root_bounds, 'child_bounds': check_child_bounds,
     'cone_grid': check_cone_grid, 'two_devices': check_two_devices}[sys.argv[1]](sys.argv[2])
    print('ok')
