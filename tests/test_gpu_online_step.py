"""Online fine-tuning inside the device-resident frontier step: gnnb_score_grad_device (device terms, inactive and
out-of-range terms, waves over the named subdomains only) and FrontierStep(online=True) against the oracle's autograd
gradients and torch.optim.Adam.

The checks that build a FrontierStep run in their own process (`_run_isolated`: python tests/test_gpu_online_step.py <check>
<arg>, exit code 0 = pass).

Gradients are float atomics summed over thread blocks in an order the hardware picks, so two runs of the same pass may differ
in the last bits: gradients that must be "the same" are held to 1e-5 of each tensor's largest entry (reassociation only);
term scores come from one block each and are compared bit for bit.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np                                               # noqa: E402
import pytest                                                    # noqa: E402
import torch                                                     # noqa: E402

from golden_io import GOLDEN, load_case, load_gnn, load_root     # noqa: E402
from gnn_branching_b200 import GraphNet                          # noqa: E402
from oracle import graphnet_oracle as O                          # noqa: E402
from oracle import online_oracle as OO                           # noqa: E402

pytestmark = pytest.mark.gpu

REASSOC = 1e-5                  # max|g - g'| <= REASSOC * max|g| per tensor: the same sums in another atomic order


def _model():
    model = GraphNet(2, 64, math='tc')
    model.load_state_dict(load_gnn('random'))
    return model.eval().cuda()


def _scorer(net):
    sc = _model().scorer(0)
    sc.set_network(net, key=net.key)
    return sc


def _terms(fr, rows):
    """Three terms per subdomain of ``rows``, as in test_score_gradients_match_oracle_batched."""
    terms = []
    for b in rows:
        cand = fr.mask[b].nonzero().view(-1).tolist()
        terms += [(b, cand[0], 1.0), (b, cand[len(cand) // 2], -0.5 - b), (b, cand[-1], 0.25)]
    return terms


def _device_terms(terms):
    dev = torch.device('cuda', 0)
    return (torch.tensor([t[0] for t in terms], dtype=torch.int32, device=dev),
            torch.tensor([t[1] for t in terms], dtype=torch.int32, device=dev),
            torch.tensor([t[2] for t in terms], dtype=torch.float32, device=dev))


def _same_grads(a, b, what):
    for k, v in a.items():
        err, scale = float((v - b[k]).abs().max()), float(v.abs().max())
        assert err <= REASSOC * scale, (what, k, err, scale)


@pytest.mark.parametrize('arch,B', [('base', 3), ('deep', 2)])
def test_device_terms_equal_host_terms(arch, B):
    fr, _ = load_case(arch, 'fr')
    fr = fr.slice(0, B).to('cuda')
    sc = _scorer(fr.net)
    terms = _terms(fr.cpu(), range(B))
    vals_host = sc.score_grad(fr, terms)
    g_host = sc.gradients()
    vals_dev = sc.score_grad(fr, _device_terms(terms))
    assert vals_dev.is_cuda
    assert torch.equal(vals_dev.cpu(), vals_host)
    assert sc.get_option('grad_workspace_domains') == B and sc.get_option('grad_bad_terms') == 0
    _same_grads(g_host, sc.gradients(), 'device terms')


def test_inactive_and_out_of_range_terms():
    fr, _ = load_case('base', 'fr')
    B = 3
    fr = fr.slice(0, B).to('cuda')
    sc = _scorer(fr.net)
    nh = fr.net.n_hidden
    terms = _terms(fr.cpu(), range(B))
    vals = sc.score_grad(fr, _device_terms(terms))
    g = sc.gradients()
    extra = [(-1, 5, 1.0), (B, 0, 1.0), (0, nh, 1.0), (-7, nh + 3, 2.0), (1, -1, 1.0), (B + 100, 3, -1.0)]
    bad = 4                                       # domain = B, index = n_hidden, index = -1, domain = B + 100
    mixed = extra[:3] + terms[:4] + extra[3:] + terms[4:]
    vals2 = sc.score_grad(fr, _device_terms(mixed)).cpu()
    assert sc.get_option('grad_bad_terms') == bad
    active = [i for i, t in enumerate(mixed) if t in terms]
    assert torch.equal(vals2[active], vals.cpu())
    assert torch.isnan(vals2[[i for i in range(len(mixed)) if i not in active]]).all()
    _same_grads(g, sc.gradients(), 'inactive terms')
    # only inactive / bad terms: no subdomain is run, the gradients are zero
    vals3 = sc.score_grad(fr, _device_terms(extra)).cpu()
    assert torch.isnan(vals3).all() and sc.get_option('grad_bad_terms') == bad and sc.get_option('grad_workspace_domains') == 0
    assert all(float(v.abs().max()) == 0.0 for v in sc.gradients().values())


def test_waves_skip_unnamed_subdomains():
    from test_gpu_parity import _assert_grads
    from gnn_branching_b200 import synthetic_frontier
    fr = synthetic_frontier(*load_root('base'), 7, seed=11)
    rows = [0, 1, 3, 4, 6]                        # subdomains 2 and 5 carry no term
    terms = _terms(fr, rows)
    ref, vals_ref = OO.score_grads(load_gnn('random'), fr, terms)
    sc = _scorer(fr.net)
    sc.set_option('grad_chunk', 2)
    vals = sc.score_grad(fr.to('cuda'), _device_terms(terms)).cpu()
    assert 1 <= sc.get_option('grad_workspace_domains') <= 2
    assert float((vals - vals_ref).abs().max()) <= 1e-5 * float(vals_ref.abs().max())
    g2 = sc.gradients()
    _assert_grads(g2, ref, rtol=2e-2)
    sc.set_option('grad_chunk', 0)
    vals0 = sc.score_grad(fr.to('cuda'), _device_terms(terms)).cpu()
    assert sc.get_option('grad_workspace_domains') == len(rows)
    assert torch.equal(vals0, vals)
    _same_grads(sc.gradients(), g2, 'waves of 2 against one wave')


def test_online_argument_errors():
    from gnn_branching_b200 import FrontierStep
    net, lbs, ubs, wp, bp = load_root('base')
    x = torch.zeros(net.n0)
    with pytest.raises(ValueError):
        FrontierStep(_model(), net, x, 0.1, wp, bp, online=True)
    with pytest.raises(ValueError):
        FrontierStep(_model(), net, x, 0.1, wp, bp, online=True, kw_fallback=True, strong_branching_k=2)
    with pytest.raises(ValueError):
        FrontierStep(_model(), net, x, 0.1, wp, bp, online=True, strong_branching_k=2)


def _iso(what, arg, timeout=300):
    from test_gpu_parity import _run_isolated
    _run_isolated(what, arg, timeout=timeout, script=os.path.basename(__file__))


def test_online_step_matches_oracle():
    _iso('online_step', 'base')


@pytest.mark.parametrize('arch', ['wide', 'deep'])
def test_online_step_other_nets(arch):
    _iso('online_nets', arch)


# ---- checks run in their own process -------------------------------------------------------------------------------------
def _online_step(arch, **kw):
    from gnn_branching_b200 import FrontierStep
    net, lbs, ubs, wp, bp = load_root(arch)
    x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))[f'{arch}_x'].copy()).reshape(-1)
    model = _model()
    fs = FrontierStep(model, net, x, 0.145, wp, bp, capacity=8192, decision_bound=float('inf'), kw_fallback=True,
                      branching_threshold=1e9, online=True, **kw)
    fs.seed_root(lbs, ubs)
    rec = {}
    pick, add = fs.queue.pick, fs.queue.add

    def rec_pick(*a, **k):
        rec['parents'] = pick(*a, **k)
        return rec['parents']

    def rec_add(d, keep=None):
        rec['kids'] = (d, keep)
        return add(d, keep=keep)
    fs.queue.pick, fs.queue.add = rec_pick, rec_add
    return fs, model, rec


def _cpu(sd):
    return {k: v.detach().cpu() for k, v in sd.items()}


def _same_weights(a, b):
    return all(torch.equal(a[k].cpu(), b[k].cpu()) for k in a)


def check_online_step(arch):
    """FrontierStep(online=True) against the oracle, step by step: the gradients of the +-1/m terms on the trained parents'
    frontier (autograd), one torch.optim.Adam step from the pre-step parameters (its state carried across steps), and the
    children's decisions under the updated weights.  A step in which KW wins nowhere takes no Adam step."""
    fs, model, rec = _online_step(arch)
    sc = fs.scorer
    lr, wd = fs.online_lr, fs.online_wd
    params = {k: torch.nn.Parameter(v.clone()) for k, v in sc.weights().items()}
    opt = torch.optim.Adam(list(params.values()), lr=lr, weight_decay=wd)
    trained = 0
    for i, B in enumerate((1, 2, None, 4, 8)):
        pre = sc.weights()
        if B is None:                               # nothing passes the threshold: no KW decision, no online update
            fs.branching_threshold = -1e9
            st = fs.step(4)
            fs.branching_threshold = 1e9
            assert st.kw_tried == 0 and st.online_trained == 0 and fs.last_online is None, st
            assert _same_weights(pre, sc.weights())
            continue
        st = fs.step(B)
        assert 0 < st.picked <= B and st.kw_tried == st.picked and st.online_trained == st.kw_used, st
        if st.online_trained == 0:
            assert fs.last_online is None and _same_weights(pre, sc.weights())
            continue
        trained += 1
        rows, gflat, kflat, vals = [t.cpu() for t in fs.last_online]
        m = st.online_trained
        assert rows.numel() == m and vals.numel() == 2 * m
        par = rec['parents']
        fr = fs._frontier(par.lb, par.ub, par.mask).cpu()
        terms = [(int(r), int(g), 1.0 / m) for r, g in zip(rows, gflat)] + [(int(r), int(k), -1.0 / m) for r, k in zip(rows, kflat)]
        grads, vals_ref = OO.score_grads(pre, fr, terms)
        assert float((vals - vals_ref).abs().max()) <= 1e-5 * float(vals_ref.abs().max()), (vals, vals_ref)
        for k, q in params.items():
            q.data.copy_(pre[k])
            q.grad = grads[k].clone()
        opt.step()
        post = sc.weights()
        worst = max(float((post[k] - q.detach()).abs().max()) for k, q in params.items())
        assert worst <= 0.05 * lr, (B, worst)
        # the children were decided by the updated GNN
        kids, keep = rec['kids']
        keep = keep.cpu()
        kfr = fs._frontier(kids.lb, kids.ub, kids.mask).cpu()
        s_or, _ = O.gnn_forward(post, kfr)
        dec = kids.decision.cpu().long()
        flat = fs.offsets.cpu()[dec[:, 0]] + dec[:, 1]
        rep = O.parity_report(s_or[keep], s_or[keep], kfr.mask[keep], flat[keep])
        assert rep['decisions_wrong'] == 0 and rep['decisions_checked'] > 0, rep
        print(f'online_step {arch}: B {B}, m {m}, Adam step within {worst / lr:.4f} lr of the oracle', flush=True)
    assert trained > 0, 'KW won on no parent: the online update was never exercised'
    # the module follows the context, and scoring uses the updated weights without a re-upload of stale ones
    w = sc.weights()
    assert _same_weights(_cpu(model.state_dict()), w)
    par = rec['parents']
    fr = fs._frontier(par.lb, par.ub, par.mask)
    _, idx, scores = model.score_frontier(fr)
    s_new, _ = O.gnn_forward(w, fr.cpu())
    rep = O.parity_report(scores.cpu(), s_new, fr.mask.cpu(), idx.cpu(), rtol=1e-4)
    assert rep['ok'], rep
    assert _same_weights(_cpu(model.state_dict()), sc.weights())


def check_online_nets(arch):
    """Several batched online steps keep the invariants of check_frontier_step (tests/gpu_isolated.py)."""
    fs, model, _ = _online_step(arch)
    glb, size, used = fs.queue.global_lb, 1, 0
    for B in (1, 2, 4, 8, 16, 32):
        st = fs.step(B)
        size += st.added - st.picked
        used += st.online_trained
        assert st.kw_tried == st.picked and st.online_trained == st.kw_used and len(fs.queue) == size, (st, size)
        assert st.children == 2 * st.picked and st.added <= st.children - st.infeasible
        assert st.global_lb >= glb - 1e-6, (st.global_lb, glb)
        glb = st.global_lb
    assert _same_weights(_cpu(model.state_dict()), fs.scorer.weights())
    print(f'online_nets {arch}: {used} parents trained on, queue {len(fs.queue)}', flush=True)


if __name__ == '__main__':
    {'online_step': check_online_step, 'online_nets': check_online_nets}[sys.argv[1]](sys.argv[2])
    print('ok')
