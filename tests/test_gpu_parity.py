"""Parity of the CUDA path (through the C ABI) with the reference's committed outputs and with the oracle.

Tolerances (BASELINE.json north_star): per subdomain max|s_new - s_ref| <= 1e-4 * max|s_ref| over candidate rows;
identical branching decision wherever the reference's top-2 margin exceeds 2e-4 * max|s_ref|.
The exact-fp32 SIMT mode is held to 1e-5.
"""
import os

import pytest
import torch

from golden_io import ARCHS, load_case, load_gnn, load_root
from gnn_branching_b200 import GraphNet, GraphChoice, Frontier, Scorer, synthetic_frontier, _lib
from gnn_branching_b200.engine import flat_to_layer_index
from oracle import graphnet_oracle as O

pytestmark = pytest.mark.gpu

MODES = ['simt', 'tc']
RTOL = {'simt': 1e-5, 'tc': 1e-4}


def _modes():
    out = []
    for m in MODES:
        out.append(m)
    return out


def _model(weights, math, T=2, chunk=0):
    model = GraphNet(T, 64, math=math, chunk=chunk)
    model.load_state_dict(load_gnn(weights))
    return model.eval().cuda()


def _skip_if_unbuilt(math):
    if math == 'tc':
        try:
            Scorer(0, math='tc')
        except _lib.GnnbError as e:
            if e.status == _lib.GNNB_ERR_UNSUPPORTED:
                pytest.skip('tensor-core path not built yet')
            raise


@pytest.mark.parametrize('math', MODES)
@pytest.mark.parametrize('weights', ['random', 'shipped'])
@pytest.mark.parametrize('case', ['fr', 'root'])
@pytest.mark.parametrize('arch', ARCHS)
def test_scores_and_decisions_match_reference(arch, case, weights, math):
    _skip_if_unbuilt(math)
    fr, ref = load_case(arch, case)
    model = _model(weights, math)
    best, idx, scores = model.score_frontier(fr.to('cuda'))
    rep = O.parity_report(scores.cpu(), ref[f'scores_{weights}'], fr.mask, idx.cpu(), rtol=RTOL[math])
    assert rep['ok'], rep
    dec = [flat_to_layer_index(int(i), fr.net.hidden_sizes) for i in idx.cpu()]
    assert dec == ref[f'decisions_{weights}'].tolist()
    # best score is the score at the winning index
    for b in range(fr.B):
        assert float(best[b]) == float(scores[b, int(idx[b])])


@pytest.mark.parametrize('math', MODES)
@pytest.mark.parametrize('T', [1, 3])
def test_other_round_counts(T, math):
    _skip_if_unbuilt(math)
    fr, ref = load_case('base', 'fr')
    model = _model('random', math, T=T)
    _, idx, scores = model.score_frontier(fr.to('cuda'))
    rep = O.parity_report(scores.cpu(), ref[f'scores_random_T{T}'], fr.mask, idx.cpu(), rtol=RTOL[math])
    assert rep['ok'], rep


@pytest.mark.parametrize('math', MODES)
@pytest.mark.parametrize('arch', ['base', 'deep'])
def test_every_stage_matches_oracle(arch, math):
    """Stage-by-stage snapshots (nb, relax, mu of every layer, both sweeps, both rounds) against the oracle."""
    _skip_if_unbuilt(math)
    fr, _ = load_case(arch, 'fr')
    sd = load_gnn('random')
    stages = {}
    O.gnn_forward(sd, fr, stages=stages)
    model = _model('random', math)
    sc = model.scorer(0)
    sc.set_option('snapshot', 1)
    model.score_frontier(fr.to('cuda'))
    tol = 2e-5 if math == 'simt' else 2e-4
    worst = {}
    for name, want in stages.items():
        key = name
        if '_relax' in name:      # relaxation features are round-independent: computed once
            if not name.startswith('t0_') or math == 'tc':
                continue          # (the tensor-core path stores them pre-multiplied by fc4 / bc4: covered through mu)
            key = name.replace('t0_fwd_relax', 'relax_f').replace('t0_bwd_relax', 'relax_b')
        got = sc.snapshot(key).reshape(want.shape)
        err = float((got - want).abs().max()) / max(float(want.abs().max()), 1e-20)
        worst[name] = err
        assert err <= tol, (name, err)
    sc.set_option('snapshot', 0)


@pytest.mark.parametrize('math', MODES)
def test_reference_api_forward_and_decision(tmp_path, math):
    """GraphNet.forward / GraphChoice.decision called exactly like the reference calls them."""
    _skip_if_unbuilt(math)
    fr, ref = load_case('base', 'root')
    model = _model('shipped', math)
    args = fr.to('cuda').to_reference_args()
    with torch.no_grad():
        ragged = model(*args)
    assert isinstance(ragged, list) and len(ragged) == fr.B
    for b in range(fr.B):
        want = ref['scores_shipped'][b][fr.mask[b].nonzero().view(-1)]
        assert ragged[b].shape == want.shape
        assert float((ragged[b].cpu() - want).abs().max()) <= RTOL[math] * float(want.abs().max())
    # GraphChoice: checkpoint file on disk, BaB mask convention (-1 undecided), B = 1, python-float primals
    ckpt = os.path.join(tmp_path, 'gnn.pt')
    torch.save(load_gnn('shipped'), ckpt)
    for b in range(fr.B):
        one = fr.slice(b, b + 1)
        lbs, ubs, duals, primals, pin, layers, masks = one.to_reference_args()
        init_mask, off = [], 0
        for n in fr.net.hidden_sizes:
            m = masks[0, off:off + n]
            init_mask.append(torch.where(m != 0, torch.full_like(m, -1), torch.ones_like(m)).int())
            off += n
        gc = GraphChoice(init_mask, ckpt, math=math)
        dec = gc.decision(lbs, ubs, duals, pin, [q.tolist() for q in primals], layers, init_mask)
        assert dec == ref['decisions_shipped'][b].tolist()


@pytest.mark.parametrize('math', MODES)
def test_host_buffers_and_chunking_give_identical_results(math):
    """mem = HOST (copies inside the call) and any chunk size must give bit-identical results to one
    device-resident chunk: subdomains are independent (SURVEY §8e)."""
    _skip_if_unbuilt(math)
    net, lbs, ubs, wp, bp = load_root('base')
    fr = synthetic_frontier(net, lbs, ubs, wp, bp, 13, seed=5)
    model = _model('random', math, chunk=13)
    b0, i0, s0 = model.score_frontier(fr.to('cuda'))
    model2 = _model('random', math, chunk=4)
    b1, i1, s1 = model2.score_frontier(fr.to('cuda'))
    assert torch.equal(s0, s1) and torch.equal(i0, i1) and torch.equal(b0, b1)
    b2, i2, s2 = model2.score_frontier(fr.pin())
    assert not s2.is_cuda
    assert torch.equal(s0.cpu(), s2) and torch.equal(i0.cpu(), i2) and torch.equal(b0.cpu(), b2)


@pytest.mark.parametrize('math', MODES)
def test_empty_candidate_set_and_nan(math):
    _skip_if_unbuilt(math)
    fr, _ = load_case('base', 'fr')
    fr.mask[1].zero_()
    model = _model('random', math)
    best, idx, _ = model.score_frontier(fr.to('cuda'))
    assert int(idx[1]) == -1 and float(best[1]) == float('-inf')
    assert int(idx[0]) >= 0
    # l = u = 0 is 0/0 in compute_ratio (graph_conv.py:502); the reference stops in pdb, the library reports it
    fr.lb[1][0, 5] = 0.0
    fr.ub[1][0, 5] = 0.0
    with pytest.raises(_lib.GnnbError) as ei:
        model.score_frontier(fr.to('cuda'))
    assert ei.value.status == _lib.GNNB_ERR_NAN
    # the flag is cleared and the context stays usable
    fr2, _ = load_case('base', 'fr')
    model.score_frontier(fr2.to('cuda'))


@pytest.mark.parametrize('math', MODES)
@pytest.mark.parametrize('arch,B', [('base', 1024), ('wide', 4096), ('deep', 4096)])
def test_full_size_frontier_properties(arch, B, math):
    """BASELINE config sizes (base x 1 024, wide x 4 096, deep x 4 096; the exact-fp32 SIMT mode runs wide / deep at 512 to bound
    the test time): oracle parity on a slice + batch invariance (a subdomain's scores do not depend on its neighbours)."""
    _skip_if_unbuilt(math)
    if math == 'simt' and B > 1024:
        B = 512
    net, lbs, ubs, wp, bp = load_root(arch)
    fr = synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=1000 * (2 + ARCHS.index(arch)), device='cuda')
    model = _model('random', math)
    best, idx, scores = model.score_frontier(fr)
    # oracle parity on 12 subdomains spread over the whole frontier (first and last wave items, ragged tail included)
    ids = torch.tensor(sorted({0, 1, B // 7, B // 3, B // 2 - 1, B // 2, (2 * B) // 3, B - 130, B - 129, B - 3, B - 2, B - 1}), device='cuda')
    sl = fr._map(lambda t: t[ids]).cpu().contiguous()
    s_or, _ = O.gnn_forward(load_gnn('random'), sl)
    rep = O.parity_report(scores[ids].cpu(), s_or, sl.mask, idx[ids].cpu(), rtol=RTOL[math])
    assert rep['ok'], rep
    b2, i2, s2 = model.score_frontier(fr.slice(B - 3, B).contiguous())
    assert torch.equal(s2, scores[B - 3:]) and torch.equal(i2, idx[B - 3:])
    # every winner is a candidate and is the masked maximum of its row
    m = fr.mask != 0
    masked = torch.where(m, scores, torch.full_like(scores, float('-inf')))
    assert torch.equal(masked.max(1).values, best)
    assert bool(m[torch.arange(B, device='cuda'), idx.long()].all())


def test_frontier_of_65536_subdomains():
    """BASELINE config 5 size on one GPU (>= 64 k CIFAR-base subdomains per call, scored in waves): every winner is a
    candidate and the masked maximum of its row; a slice scored on its own gives bit-identical results."""
    B = 65536
    net, lbs, ubs, wp, bp = load_root('base')
    model = _model('random', 'tc')
    fr = synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=424242, device='cuda')
    best, idx, _ = model.score_frontier(fr, return_scores=False)
    assert best.shape == (B,) and idx.shape == (B,)
    assert bool((idx >= 0).all()) and bool(torch.isfinite(best).all())
    m = fr.mask != 0
    assert bool(m[torch.arange(B, device='cuda'), idx.long()].all())
    for start in (0, 40000, B - 5):
        sl = fr.slice(start, start + 5).contiguous()
        b2, i2, s2 = model.score_frontier(sl, return_scores=True)
        assert torch.equal(b2, best[start:start + 5]) and torch.equal(i2, idx[start:start + 5])
        masked = torch.where(sl.mask != 0, s2, torch.full_like(s2, float('-inf')))
        assert torch.equal(masked.max(1).values, b2)
    # oracle parity on 10 subdomains spread over the 64 waves
    ids = torch.tensor([0, 1023, 1024, 20000, 32767, 32768, 50001, B - 1025, B - 2, B - 1], device='cuda')
    pick = fr._map(lambda t: t[ids].contiguous())
    sl = pick.cpu().contiguous()
    s_or, _ = O.gnn_forward(load_gnn('random'), sl)
    b3, i3, s3 = model.score_frontier(pick)
    assert torch.equal(b3, best[ids]) and torch.equal(i3, idx[ids])
    rep = O.parity_report(s3.cpu(), s_or, sl.mask, i3.cpu(), rtol=RTOL['tc'])
    assert rep['ok'], rep


@pytest.mark.parametrize('arch', ARCHS)
def test_fused_layer_kernel_matches_two_launches(arch):
    """The default path (option fuse = 1: propagation gather-GEMM and node-update chain of a layer in one kernel, nb handed
    over in tensor memory) against the two-launch path (fuse = 0, nb through HBM): both split the same fp32 accumulator into
    the same fp16 hi / lo operand; the first chain GEMM reads it from tensor memory instead of shared memory, which changes the
    hardware's accumulation order (1.3e-6 of the largest score measured) — held to 1e-5 — and both match the reference."""
    from gpu_isolated import _close
    fr, ref = load_case(arch, 'fr')
    model = _model('random', 'tc')
    sc = model.scorer(0)
    assert sc.get_option('fuse') == 1
    b1, i1, s1 = model.score_frontier(fr.to('cuda'))
    sc.set_option('fuse', 0)
    b0, i0, s0 = model.score_frontier(fr.to('cuda'))
    _close(s0, s1, i0, i1, fr.mask.cuda(), f'{arch} golden frontier')
    for s_, i_ in ((s0, i0), (s1, i1)):
        rep = O.parity_report(s_.cpu(), ref['scores_random'], fr.mask, i_.cpu(), rtol=RTOL['tc'])
        assert rep['ok'], rep
    net, lbs, ubs, wp, bp = load_root(arch)
    big = synthetic_frontier(net, lbs, ubs, wp, bp, 301, seed=77, device='cuda')     # several items per CTA, a ragged last group
    b2, i2, s2 = model.score_frontier(big)
    sc.set_option('fuse', 1)
    b3, i3, s3 = model.score_frontier(big)
    _close(s2, s3, i2, i3, big.mask, f'{arch} x 301')


def _custom_frontier(layers, input_shape, B, seed):
    from torch import nn
    from gnn_branching_b200 import netspec_from_modules
    from gnn_branching_b200.frontier import interval_root_bounds
    g = torch.Generator().manual_seed(seed)
    for m in layers:
        for q in m.parameters():
            q.data = torch.randn(q.shape, generator=g) * (0.3 if q.dim() > 1 else 0.1)
    net = netspec_from_modules(layers, input_shape, name='custom')
    x = torch.randn(input_shape, generator=g)
    wp = torch.randn(net.hidden_sizes[-1], generator=g) * 0.3
    lbs, ubs = interval_root_bounds(net, x.reshape(-1), 0.05, wp, 0.1)
    return synthetic_frontier(net, lbs, ubs, wp, 0.1, B, seed=seed, max_splits=4)


@pytest.mark.parametrize('math', MODES)
@pytest.mark.parametrize('case', ['odd_shapes', 'wide_channels', 'deep_narrow'])
def test_other_network_shapes_match_oracle(case, math):
    """Networks that are not the three CIFAR ones: odd spatial sizes and channel counts (padding slots in every tile),
    more than 128 channels (channel-blocked tiles), 3x3 / 5x5 kernels, stride 1 and 2 — against the oracle."""
    from torch import nn
    from gnn_branching_b200 import Flatten
    if case == 'odd_shapes':
        layers = [nn.Conv2d(2, 5, 3, stride=1, padding=1), nn.ReLU(), nn.Conv2d(5, 6, 3, stride=2, padding=1), nn.ReLU(),
                  Flatten(), nn.Linear(6 * 5 * 4, 37), nn.ReLU()]
        shape, B = (2, 9, 7), 7
    elif case == 'wide_channels':
        layers = [nn.Conv2d(3, 130, 3, stride=1, padding=1), nn.ReLU(), Flatten(), nn.Linear(130 * 4 * 4, 20), nn.ReLU()]
        shape, B = (3, 4, 4), 5
    else:
        layers = [nn.Conv2d(1, 4, 5, stride=1, padding=2), nn.ReLU(), nn.Conv2d(4, 4, 3, stride=1, padding=1), nn.ReLU(),
                  nn.Conv2d(4, 3, 4, stride=2, padding=1), nn.ReLU(), Flatten(), nn.Linear(3 * 6 * 6, 150), nn.ReLU(),
                  nn.Linear(150, 9), nn.ReLU()]
        shape, B = (1, 12, 12), 6
    fr = _custom_frontier(layers, shape, B, seed=11)
    sd = load_gnn('random')
    s_or, _ = O.gnn_forward(sd, fr)
    model = _model('random', math)
    best, idx, scores = model.score_frontier(fr.to('cuda'))
    rep = O.parity_report(scores.cpu(), s_or, fr.mask, idx.cpu(), rtol=RTOL[math])
    assert rep['ok'], rep
    if math == 'tc':
        from gpu_isolated import _close
        model.scorer(0).set_option('fuse', 0)
        b1, i1, s1 = model.score_frontier(fr.to('cuda'))
        _close(s1, scores, i1, idx, fr.mask.cuda(), case)


# ---- BaBSR / KW heuristic (SURVEY §8f rank 1) -------------------------------------------------------------------
@pytest.mark.parametrize('case', ['fr', 'root'])
@pytest.mark.parametrize('arch', ARCHS)
def test_babsr_matches_reference(arch, case):
    """gnnb_babsr against the reference's choose_node_conv outputs: scores to 1e-5 of the largest score, decisions and
    counters exactly, in the three branches of the decision rule; device and host buffers agree."""
    import numpy as np
    from golden_io import GOLDEN
    from gnn_branching_b200 import babsr_frontier
    z = dict(np.load(os.path.join(GOLDEN, f'babsr_{arch}.npz')))
    fr, _ = load_case(arch, case)
    order = [0] + [k for k in range(fr.net.L) if k != 0]
    ref = torch.from_numpy(z[f'{case}_scores'])
    for name, (thr, cnt) in {'score': (0.001, 0), 'intercept': (1e9, 0), 'order': (1e9, 2)}.items():
        dec, cout, kind, scores = babsr_frontier(fr.to('cuda'), [cnt] * fr.B, order, 0, thr, return_scores=True)
        assert float((scores.cpu() - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
        assert dec.cpu().tolist() == z[f'{case}_{name}_decisions'].tolist()
        assert cout.cpu().tolist() == z[f'{case}_{name}_counters'].tolist()
        assert kind.cpu().tolist() == [{'score': 0, 'intercept': 1, 'order': 2}[name]] * fr.B
        d2, c2, k2, s2 = babsr_frontier(fr.contiguous(), [cnt] * fr.B, order, 0, thr, return_scores=True)
        assert not d2.is_cuda and torch.equal(d2, dec.cpu()) and torch.equal(c2, cout.cpu()) and torch.equal(s2, scores.cpu())


@pytest.mark.parametrize('arch,B', [('base', 1024), ('deep', 257)])
def test_babsr_frontier_matches_oracle(arch, B):
    """A whole synthetic frontier: scores against the oracle, decisions equal wherever the oracle's top-2 margin
    exceeds the tolerance; the reference-signature wrapper agrees on single subdomains."""
    from gnn_branching_b200 import babsr_frontier, choose_node_conv
    from oracle import babsr_oracle as BO
    net, lbs, ubs, wp, bp = load_root(arch)
    fr = synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=31, device='cuda')
    order = [0] + [k for k in range(net.L) if k != 0]
    dec, cout, kind, scores = babsr_frontier(fr, None, order, 0, 0.001, return_scores=True)
    fc = fr.cpu().contiguous()
    sc, ic = BO.babsr_scores(fc)
    tol = 1e-5 * float(sc.abs().max())
    assert float((scores.cpu() - sc).abs().max()) <= tol
    d_or, c_or, k_or = BO.babsr_decide(sc, ic, fc.mask, net.hidden_sizes, [0] * B, order, 0, 0.001)
    top2 = sc.topk(2, dim=1).values
    safe = (top2[:, 0] - top2[:, 1]) > 2 * tol
    assert int(safe.sum()) > B // 2
    assert torch.equal(dec.cpu()[safe].long(), d_or[safe]) and torch.equal(cout.cpu()[safe].long(), c_or[safe])
    # reference-signature call, B = 1
    one = fc.slice(3, 4)
    lbs1, ubs1, _, _, _, layers, masks = one.to_reference_args()
    modules = layers['fixed_layers'] + [layers['prop_layers'][0]]
    pre_relu = list(range(1, net.L + 1))
    init_mask, off = [], 0
    for n in net.hidden_sizes:
        m = masks[0, off:off + n]
        init_mask.append(torch.where(m != 0, torch.full_like(m, -1), torch.ones_like(m)).int())
        off += n
    d1, c1 = choose_node_conv([t[0] for t in lbs1], [t[0] for t in ubs1], init_mask, modules, pre_relu, 0, order, 0)
    assert d1 == dec[3].tolist() and c1 == int(cout[3])


# ---- online fine-tuning (SURVEY §8f rank 2) -----------------------------------------------------------------------
# per tensor: max|g - g_ref| <= GRAD_RTOL * max|g_ref| + GRAD_ATOL.  Both sides are fp32 sums over thousands of rows in
# different orders; the absolute floor (5 ulp of the O(1) scores being differentiated) covers tensors at the end of the
# longest chains (inp_f on the 5-layer net: |g| ~ 1e-4 after cancellation, observed difference 1.3e-7)
GRAD_RTOL, GRAD_ATOL = 1e-4, 3e-7


def _bab_mask(fr, b):
    out, off = [], 0
    for n in fr.net.hidden_sizes:
        m = fr.mask[b, off:off + n]
        out.append(torch.where(m != 0, torch.full_like(m, -1), torch.ones_like(m)).int())
        off += n
    return out


def _flat(fr, dec):
    return sum(fr.net.hidden_sizes[:dec[0]]) + dec[1]


def _assert_grads(got, ref, rtol=GRAD_RTOL):
    for k, r in ref.items():
        err, scale = float((got[k] - r).abs().max()), float(r.abs().max())
        assert err <= rtol * scale + GRAD_ATOL, (k, err, scale)


@pytest.mark.parametrize('weights', ['random', 'shipped'])
def test_score_gradients_match_reference(weights):
    """gnnb_score_grad against the reference's own p.grad after loss.backward() (graph_score_online.py:74-75)."""
    from golden_io import load_online
    z = load_online()
    fr, _ = load_case('base', 'fr')
    one = fr.slice(0, 1).to('cuda')
    model = _model(weights, 'tc')
    sc = model.scorer(0)
    sc.set_network(fr.net, key=fr.net.key)
    gnn, kw = _flat(fr, z[f'{weights}_dec0'].tolist()), _flat(fr, z[f'{weights}_kw0'].tolist())
    vals = sc.score_grad(one, [(0, gnn, 1.0), (0, kw, -1.0)])
    assert abs(float(vals[0]) - float(z[f'{weights}_gnn_score0'])) <= 1e-5 * abs(float(z[f'{weights}_gnn_score0']))
    assert abs(float(vals[1]) - float(z[f'{weights}_kw_score0'])) <= 1e-5 * max(1.0, abs(float(z[f'{weights}_kw_score0'])))
    ref = {k: torch.from_numpy(z[f'{weights}_grad0_{k}']) for k in sc.gradients()}
    _assert_grads(sc.gradients(), ref)


@pytest.mark.parametrize('arch,B', [('deep', 2), ('wide', 2), ('base', 3)])
def test_score_gradients_match_oracle_batched(arch, B):
    """Several subdomains and terms at once, other network shapes (3x3 stride-1 convs, 5 hidden layers), host buffers.

    Tolerance 2e-2 per tensor: a gradient through ~30 ReLU layers is a discontinuous function of the fp32 rounding of the
    forward pass — a pre-activation within one ulp of zero gives a different ReLU mask in two equally valid fp32
    evaluations, and one flipped unit moves the gradients behind it by 1e-3 .. 1e-2 of their size.  scripts/grad_diag.py
    measures it against an fp64 autograd oracle: where no unit flips the CUDA path is within 1e-6..3e-6 of fp64 (like
    torch's own fp32 autograd); on deep x 1 torch-fp32 itself is 6.8e-3 away from fp64; on deep x 2 the CUDA path is 5e-3
    away and torch-fp32 2e-6.  The tight bound (1e-4) is held by test_score_gradients_match_reference."""
    from oracle import online_oracle as OO
    fr, _ = load_case(arch, 'fr')
    fr = fr.slice(0, B)
    sd = load_gnn('random')
    terms = []
    for b in range(B):
        cand = fr.mask[b].nonzero().view(-1).tolist()
        terms += [(b, cand[0], 1.0), (b, cand[len(cand) // 2], -0.5 - b), (b, cand[-1], 0.25)]
    ref, vals_ref = OO.score_grads(sd, fr, terms)
    model = _model('random', 'tc')
    sc = model.scorer(0)
    sc.set_network(fr.net, key=fr.net.key)
    for dev in ('cuda', 'cpu'):
        vals = sc.score_grad(fr.to(dev), terms)
        assert float((vals - vals_ref).abs().max()) <= 1e-5 * float(vals_ref.abs().max())
        _assert_grads(sc.gradients(), ref, rtol=2e-2)


def test_online_learning_matches_reference(tmp_path):
    """graph_score_online.GraphChoice used exactly like plnn/relu_conv_online.py uses the reference: decision, online_learning
    against a KW decision, twice; decisions equal the reference's, the parameters after two Adam steps agree to a small
    fraction of one step (Adam's step is lr * m / (sqrt(v) + eps): O(lr) per element whatever the gradient's size)."""
    from golden_io import load_online
    from gnn_branching_b200.graph_score_online import GraphChoice as OnlineChoice
    z = load_online()
    lr, wd = float(z['lr']), float(z['wd'])
    fr, _ = load_case('base', 'fr')
    ckpt = os.path.join(tmp_path, 'gnn.pt')
    torch.save(load_gnn('random'), ckpt)
    gc = OnlineChoice(_bab_mask(fr, 0), ckpt, lr=lr, wd=wd)
    for step in (0, 1):
        one = fr.slice(step, step + 1)
        lbs, ubs, duals, primals, pin, layers, _ = one.to_reference_args()
        dec = gc.decision(lbs, ubs, duals, pin, [q.tolist() for q in primals], layers, _bab_mask(fr, step))
        assert dec == z[f'random_dec{step}'].tolist()
        assert abs(gc.gnn_score - float(z[f'random_gnn_score{step}'])) <= 1e-4 * abs(float(z[f'random_gnn_score{step}']))
        loss = gc.online_learning(z[f'random_kw{step}'].tolist(), 1)
        ref_loss = float(z[f'random_gnn_score{step}']) - float(z[f'random_kw_score{step}']) + 1.0
        assert abs(loss - ref_loss) <= 1e-4 * abs(ref_loss)
        gc.del_score()
    sd = gc.model.state_dict()
    worst = 0.0
    for k, v in sd.items():
        ref = torch.from_numpy(z[f'random_sd2_{k}'])
        worst = max(worst, float((v.cpu() - ref).abs().max()))
    assert worst <= 0.05 * lr, worst
    # the module and the device context hold the same parameters, and scoring uses them
    dev = gc.model.scorer(0).weights()
    for k, v in sd.items():
        assert torch.equal(v.cpu(), dev[k])
    s_new, _ = O.gnn_forward({k: v.cpu() for k, v in sd.items()}, fr)
    _, idx, scores = gc.model.score_frontier(fr.to('cuda'))
    rep = O.parity_report(scores.cpu(), s_new, fr.mask, idx.cpu(), rtol=1e-4)
    assert rep['ok'], rep


def test_adam_step_matches_torch():
    """gnnb_adam_step against torch.optim.Adam on identical gradients, three steps (bias correction, weight decay)."""
    fr, _ = load_case('base', 'fr')
    one = fr.slice(0, 1).to('cuda')
    model = _model('random', 'tc')
    sc = model.scorer(0)
    sc.set_network(fr.net, key=fr.net.key)
    params = {k: torch.nn.Parameter(v.clone()) for k, v in load_gnn('random').items()}
    opt = torch.optim.Adam(list(params.values()), lr=3e-4, weight_decay=1e-3)
    cand = fr.mask[0].nonzero().view(-1).tolist()
    for step in range(3):
        sc.score_grad(one, [(0, cand[step], 1.0), (0, cand[-1 - step], -1.0)])
        g = sc.gradients()
        for k, q in params.items():
            q.grad = g[k].clone()
        opt.step()
        sc.adam_step(3e-4, weight_decay=1e-3)
        w = sc.weights()
        for k, q in params.items():
            assert float((w[k] - q.detach()).abs().max()) <= 2e-7 + 1e-3 * 3e-4, k
            q.data.copy_(w[k])          # keep the two trajectories on the same parameters


# ---- device-resident domain queue (SURVEY §8f rank 4) ---------------------------------------------------------------
def _queue_batch(net, lbs, ids, device='cuda'):
    """Domains whose payload encodes their id: bounds row = id + layer/column pattern, mask = id % 3 - 1, decision = (id, 2 id)."""
    from gnn_branching_b200 import DomainBatch
    B = len(lbs)
    ids_t = torch.tensor(ids, dtype=torch.float32)
    sizes = [net.n0] + net.hidden_sizes + [1]
    lb = [ids_t.reshape(B, 1) + 0.001 * k + 1e-6 * torch.arange(n).reshape(1, n) for k, n in enumerate(sizes)]
    ub = [t + 0.5 for t in lb]
    mask = ((torch.tensor(ids).reshape(B, 1) + torch.arange(net.n_hidden).reshape(1, -1)) % 3 - 1).to(torch.int8)
    dec = torch.tensor([[i % 7, 2 * i] for i in ids], dtype=torch.int32)
    return DomainBatch(torch.tensor(lbs, dtype=torch.float32), torch.tensor(lbs, dtype=torch.float32) + 1.0, lb, ub, mask, dec).to(device)


def _check_payload(net, b, ids):
    ref = _queue_batch(net, [float(x) for x in b.lower_bound.cpu()], ids, device='cpu')
    got = b.to('cpu')
    assert torch.equal(got.upper_bound, ref.upper_bound)
    for k in range(len(ref.lb)):
        assert torch.equal(got.lb[k], ref.lb[k]) and torch.equal(got.ub[k], ref.ub[k])
    assert torch.equal(got.mask, ref.mask) and torch.equal(got.decision, ref.decision)


@pytest.mark.parametrize('host', [False, True])
def test_domain_queue_replays_reference_traces(host):
    """gnnb_queue_* on the reference's own traces (tests/golden/queue_traces.npz): every pick returns the domain the
    reference's pick_out returned, with its payload intact; the list left at the end is the reference's, in order."""
    import numpy as np
    from golden_io import GOLDEN
    from gnn_branching_b200 import DomainQueue
    z = dict(np.load(os.path.join(GOLDEN, 'queue_traces.npz')))
    fr, _ = load_case('base', 'fr')
    sc = Scorer(0)
    sc.set_network(fr.net, key=fr.net.key)
    dev = 'cpu' if host else 'cuda'
    for t in range(6):
        ops = z[f't{t}_ops']
        if host and len(ops) > 500:
            continue
        q = DomainQueue(sc, capacity=1024)
        picked = []
        for kind, value, ident in ops:
            kind = int(kind)
            if kind == 0:
                assert q.add(_queue_batch(fr.net, [float(value)], [int(ident)], device=dev)) == 1
            elif kind == 1:
                if len(q) == 0:
                    picked.append(-1)
                    continue
                b = q.pick(1, float(value), device=dev, discard_rest=True)
                if b.B == 0:
                    picked.append(-1)
                    assert len(q) == 0
                else:
                    ident_got = int(b.decision[0, 1]) // 2
                    picked.append(ident_got)
                    _check_payload(fr.net, b, [ident_got])
            else:
                q.prune(float(value))
        assert picked == z[f't{t}_picked'].tolist()
        left = z[f't{t}_left'].tolist()
        assert len(q) == len(left)
        if left:
            rest = q.pick(len(left), float('inf'), device=dev)
            assert [int(x) // 2 for x in rest.decision[:, 1].cpu()] == left
            _check_payload(fr.net, rest, left)


def test_domain_queue_batched_ops_match_oracle():
    """Batched adds (with a keep mask), picks of many domains at once and prunes against the oracle; more adds than the
    capacity raise; slots are recycled."""
    from oracle.queue_oracle import QueueOracle
    from gnn_branching_b200 import DomainQueue
    fr, _ = load_case('base', 'fr')
    sc = Scorer(0)
    sc.set_network(fr.net, key=fr.net.key)
    q, o = DomainQueue(sc, capacity=600), QueueOracle()
    g = torch.Generator().manual_seed(5)
    nid = 0
    for rnd in range(12):
        B = 150
        lbs = (torch.round(torch.randn(B, generator=g) * 8) / 8 - 1.0).tolist()
        keep = (torch.rand(B, generator=g) < 0.7)
        ids = list(range(nid, nid + B)); nid += B
        added = q.add(_queue_batch(fr.net, lbs, ids), keep=keep.cuda())
        for b in range(B):
            if keep[b]:
                o.add(lbs[b], ids[b])
        assert added == int(keep.sum()) and len(q) == len(o.domains)
        assert q.global_lb == o.domains[0].lower_bound
        thr = float(torch.randn(1, generator=g)) * 0.5 - 0.8
        want = []
        for _ in range(90):                          # pick(90) == 90 x pick_out while domains below the threshold remain
            if not o.domains or o.domains[0].lower_bound >= thr:
                break
            want.append(o.pick(thr))
        b = q.pick(90, thr)
        assert [int(x) // 2 for x in b.decision[:, 1].cpu()] == want
        _check_payload(fr.net, b, want)
        if rnd % 3 == 2:
            pt = float(torch.randn(1, generator=g)) * 0.5
            q.prune(pt); o.prune(pt)
        assert len(q) == len(o.domains)
    rest = q.pick(len(q), float('inf'))
    assert [int(x) // 2 for x in rest.decision[:, 1].cpu()] == [i for _, i in o.state()]
    with pytest.raises(_lib.GnnbError):
        q.add(_queue_batch(fr.net, [0.0] * 601, list(range(601))))


def test_domain_queue_reference_function_api():
    """add_domain / pick_out / prune_domains / domains[0].lower_bound called like plnn/relu_conv_gnnkwthreshold.py:126-244."""
    from gnn_branching_b200.domain_queue import DomainQueue, ReLUDomain, add_domain, pick_out, prune_domains
    fr, _ = load_case('base', 'fr')
    sc = Scorer(0)
    sc.set_network(fr.net, key=fr.net.key)
    domains = DomainQueue(sc, capacity=16)
    lbs, ubs, _, _, _, _, _ = fr.slice(0, 1).to_reference_args()
    mask = _bab_mask(fr, 0)
    for lb, dec in ((-0.5, [1, 7]), (-2.0, [0, 3]), (-0.5, [2, 9]), (0.3, [0, 0])):
        add_domain(ReLUDomain(mask, lb=lb, ub=1.0, lb_all=[t[0] for t in lbs], up_all=[t[0] for t in ubs], gnn_decision=dec), domains)
    assert len(domains) == 4 and domains[0].lower_bound == -2.0
    d = pick_out(domains, 0.0)
    assert d.lower_bound == -2.0 and d.gnn_decision == [0, 3] and d.upper_bound == 1.0
    assert all(torch.equal(a.cpu(), b[0]) for a, b in zip(d.lower_all, lbs)) and all(torch.equal(a.cpu(), m) for a, m in zip(d.mask, mask))
    assert pick_out(domains, 0.0).gnn_decision == [2, 9]          # equal lower bounds: the newest first (insort_left)
    domains = prune_domains(domains, 0.0)
    assert len(domains) == 1 and domains[0].lower_bound == -0.5
    assert pick_out(domains, 0.0).gnn_decision == [1, 7]
    with pytest.raises(AssertionError):
        pick_out(domains, 0.0)


_ISO_TIMED_OUT = set()


def _run_isolated(what, arg, timeout=120, env=None, script='gpu_isolated.py'):
    """Run a check of ``script`` (in tests/) in its own process (its own CUDA context) with a timeout: a hang or a sticky CUDA
    error there cannot take the rest of the suite with it.  After one time-out of a kind of check the others of that kind fail
    at once."""
    import subprocess
    import sys
    if (script, what) in _ISO_TIMED_OUT:
        pytest.fail(f'{what}: an earlier isolated check timed out')
    here = os.path.dirname(os.path.abspath(__file__))
    try:
        r = subprocess.run([sys.executable, os.path.join(here, script), what, arg], capture_output=True, text=True, timeout=timeout,
                           env=dict(os.environ, **(env or {})))
    except subprocess.TimeoutExpired:
        _ISO_TIMED_OUT.add((script, what))
        raise
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])


@pytest.mark.parametrize('math', ['0', '1'])
@pytest.mark.parametrize('arch', ARCHS)
def test_kw_bounds_match_reference(arch, math):
    """math 0: the dense layers' column blocks on the tensor-core propagation kernel (fp16 x 3), 1: exact-fp32 kernels."""
    _run_isolated('kw_bounds', arch, timeout=180, env={'GNNB_TEST_MATH': math})


@pytest.mark.parametrize('math', ['0', '1'])
@pytest.mark.parametrize('arch', ARCHS)
def test_child_bounds_match_reference_update_the_model(arch, math):
    _run_isolated('child_bounds', arch, timeout=240, env={'GNNB_TEST_MATH': math})


@pytest.mark.parametrize('arch', ['base', 'deep'])
def test_frontier_step_is_made_of_its_pieces(arch):
    _run_isolated('frontier_step', arch, timeout=240)


@pytest.mark.parametrize('math', ['0', '1'])
@pytest.mark.parametrize('case', ['odd_shapes', 'deep_narrow'])
def test_child_bounds_other_network_shapes(case, math):
    _run_isolated('child_bounds_shapes', case, timeout=240, env={'GNNB_TEST_MATH': math})
