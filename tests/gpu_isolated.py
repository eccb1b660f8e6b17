"""Checks executed in their own process (own CUDA context, time-out) by tests/test_gpu_parity.py (`_run_isolated`):
exit code 0 = pass.  Usage: python tests/gpu_isolated.py <check> <arg>"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch                                                     # noqa: E402

from golden_io import load_case, load_gnn, load_root             # noqa: E402
from gnn_branching_b200 import GraphNet, synthetic_frontier      # noqa: E402


def check_fused(arch):
    """k_tc_fused (default) against the two-launch path: both split the same fp32 propagation accumulator into the same fp16
    hi / lo operand, but the first chain GEMM reads it from tensor memory instead of shared memory and the hardware's
    accumulation order differs (measured 1.3e-6 of the largest score) — held to 1e-5, winners equal wherever the top-2 margin
    exceeds that; B chosen so that CTAs walk several items, the last group of 4 subdomains is ragged, and (B = 1) most of the
    grid is idle."""
    model = GraphNet(2, 64, math='tc')
    model.load_state_dict(load_gnn('random'))
    model = model.eval().cuda()
    sc = model.scorer(0)
    for B in (3, 1, 301, 1024):
        f = synthetic_frontier(*load_root(arch), B, seed=5 + B, device='cuda')
        sc.set_option('fuse', 1)
        b1, i1, s1 = model.score_frontier(f)
        torch.cuda.synchronize()
        sc.set_option('fuse', 0)
        b0, i0, s0 = model.score_frontier(f)
        torch.cuda.synchronize()
        _close(s0, s1, i0, i1, f.mask, f'fused {arch} B={B}')


def _close(s0, s1, i0, i1, mask, what, rtol=1e-5):
    scale = float(s0.abs().max())
    err = float((s0 - s1).abs().max()) / scale
    masked = torch.where(mask != 0, s0, torch.full_like(s0, float('-inf')))
    top2 = masked.topk(2, dim=1).values
    safe = (top2[:, 0] - top2[:, 1]) > 2 * rtol * scale
    print(f'{what}: identical={torch.equal(s0, s1)} max rel diff {err:.3e}, winners compared {int(safe.sum())}/{len(safe)}', flush=True)
    assert err <= rtol, f'{what}: scores differ by {err:.3e} of the largest score'
    assert torch.equal(i0[safe], i1[safe]), f'{what}: winners differ'


def check_kw_bounds(arch):
    """gnnb_kw_bounds against the reference's own DualNetwork: root bounds of the net (tests/golden/nets.npz) and child domains
    with one ReLU fixed, all children in one batched call (tests/golden/kw_children.npz); 5e-5 of the largest bound."""
    import numpy as np
    from golden_io import GOLDEN
    from gnn_branching_b200 import Scorer
    from oracle import kw_bounds_oracle as KW
    net, lbs, ubs, wp, bp = load_root(arch)
    x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))[f'{arch}_x'].copy()).reshape(1, -1)
    sc = Scorer(0)
    sc.set_network(net, key=net.key)
    sc.set_option('math', int(os.environ.get('GNNB_TEST_MATH', '0')))      # 0: dense layers on the tensor cores, 1: exact-fp32 kernels

    def err(a, b):
        return float((a.reshape(-1).cpu() - b.reshape(-1)).abs().max()) / max(1.0, float(b.abs().max()))

    gl, gu = sc.kw_bounds(x, 0.145, wp.reshape(1, -1), torch.tensor([bp]))
    for k in range(net.L + 2):
        assert err(gl[k], lbs[k]) <= 5e-5 and err(gu[k], ubs[k]) <= 5e-5, ('root', k, err(gl[k], lbs[k]), err(gu[k], ubs[k]))
    z = dict(np.load(os.path.join(GOLDEN, 'kw_children.npz')))
    nc = int(z[f'{arch}_ncases'])
    plbs, pubs = [], []
    for c in range(nc):
        lay, idx, choice = z[f'{arch}_c{c}_decision'].tolist()
        a, b = KW.split_bounds(lbs, ubs, (lay, idx), choice)
        plbs.append(a); pubs.append(b)
    plb = [torch.stack([plbs[c][k] for c in range(nc)]) for k in range(net.L)]
    pub = [torch.stack([pubs[c][k] for c in range(nc)]) for k in range(net.L)]
    gl, gu = sc.kw_bounds(x, 0.145, wp.reshape(1, -1).repeat(nc, 1), torch.full((nc,), float(bp)), plb, pub)
    for c in range(nc):
        for k in range(1, net.L + 2):
            rl, ru = torch.from_numpy(z[f'{arch}_c{c}_lb{k}']), torch.from_numpy(z[f'{arch}_c{c}_ub{k}'])
            l, u = gl[k][c].cpu(), gu[k][c].cpu()
            if k == net.L + 1:                     # init_kw_bounds :285-286 intersects the output bounds with the parent's
                l, u = torch.max(l, lbs[-1]), torch.min(u, ubs[-1])
            assert err(l, rl) <= 5e-5 and err(u, ru) <= 5e-5, ('child', c, k, err(l, rl), err(u, ru))


def check_child_bounds(arch):
    """gnnb_child_bounds against the UNMODIFIED reference's update_the_model (bounds part; tests/golden/child_bounds.npz): every
    golden child in ONE batched call, each from its own parent's bounds (root, child or grandchild), different split layers in
    the same batch; bounds within 5e-5 of the largest bound, the BaB mask from the rule of conv_kwinter_gen.py:696-713, the
    second-KW-pass flags equal to the reference's.  Then the same batch replicated to 64 domains (several column passes)."""
    import numpy as np
    from golden_io import GOLDEN
    from gnn_branching_b200 import Scorer
    z = dict(np.load(os.path.join(GOLDEN, 'child_bounds.npz')))
    net, _, _, wp, bp = load_root(arch)
    x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))[f'{arch}_x'].copy()).reshape(1, -1)
    L, nc = net.L, int(z[f'{arch}_ncases'])
    sc = Scorer(0)
    sc.set_network(net, key=net.key)
    sc.set_option('math', int(os.environ.get('GNNB_TEST_MATH', '0')))      # 0: dense layers on the tensor cores, 1: exact-fp32 kernels

    def get(c):
        lbs = [x[0] - 0.145] + [torch.from_numpy(z[f'{arch}_c{c}_lb{k}'].copy()) for k in range(1, L + 2)]
        ubs = [x[0] + 0.145] + [torch.from_numpy(z[f'{arch}_c{c}_ub{k}'].copy()) for k in range(1, L + 2)]
        return lbs, ubs

    def err(a, b):
        return float((a.reshape(-1).cpu() - b.reshape(-1)).abs().max()) / max(1.0, float(b.abs().max()))

    # the root first: gnnb_root_bounds against the bounds the reference's build_the_model had computed when it reached Gurobi
    # (KW bounds, interval pass from the input box, KW pass from the first layer that moved by more than 1e-4: layer 2 on all
    # three nets)
    rl, ru, rmask, rsecond = sc.root_bounds(x, 0.145, wp.reshape(1, -1), torch.tensor([bp]))
    torch.cuda.synchronize()
    gl0, gu0 = get(0)
    for k in range(L + 2):
        e = max(err(rl[k][0], gl0[k]), err(ru[k][0], gu0[k]))
        assert e <= 5e-5, ('root', k, e)
    assert int(rsecond[0]) == 1, 'the reference repeats the KW pass at the root of this net (initial kw: change_idx at 3)'
    # largest interval gain on a hidden layer after the first KW pass, per case (CPU, oracle pieces)
    from oracle import kw_bounds_oracle as KW
    gains = {}
    for c in range(1, nc):
        lay, idx, choice = z[f'{arch}_c{c}_decision'].tolist()
        lbs, ubs = get(int(z[f'{arch}_c{c}_parent']))
        (ubs if choice == 0 else lbs)[lay + 1][idx] = 0
        lbs, ubs = KW._kw_pass(net, x[0], 0.145, wp, bp, lbs, ubs, keep_upto=lay + 1)
        g = 0.0
        for k in range(lay + 2, L + 1):
            lo, hi = KW.interval_layer(net.affine[k - 1], lbs[k - 1].clamp(min=0), ubs[k - 1].clamp(min=0))
            g = max(g, float(((lo - lbs[k]) / lbs[k].abs().clamp(min=1)).max()), float(((ubs[k] - hi) / ubs[k].abs().clamp(min=1)).max()))
            lbs[k], ubs[k] = torch.max(lbs[k], lo), torch.min(ubs[k], hi)
        gains[c] = g
    for rep in (1, 64 // (nc - 1) + 1):
        cases = list(range(1, nc)) * rep
        B = len(cases)
        parents = [get(int(z[f'{arch}_c{c}_parent'])) for c in cases]
        plb = [torch.stack([p[0][k] for p in parents]) for k in range(L + 2)]
        pub = [torch.stack([p[1][k] for p in parents]) for k in range(L + 2)]
        dec = torch.tensor([z[f'{arch}_c{c}_decision'].tolist() for c in cases], dtype=torch.int32)
        gl, gu, masks, second = sc.child_bounds(x, 0.145, wp.reshape(1, -1).repeat(B, 1), torch.full((B,), float(bp)), plb, pub,
                                                dec[:, 0], dec[:, 1], dec[:, 2])
        torch.cuda.synchronize()
        worst = 0.0
        for i, c in enumerate(cases):
            rl, ru = get(c)
            for k in range(0, L + 2):
                e = max(err(gl[k][i], rl[k]), err(gu[k][i], ru[k]))
                worst = max(worst, e)
                assert e <= 5e-5, ('child', c, k, e)
            gain = gains[c]        # the library repeats the KW pass for interval gains above rounding only (gnnb_kw.cu)
            if gain > 1e-5 or gain < 1e-7:
                assert int(second[i]) == int(gain > 1e-5), ('second pass', c, int(second[i]), gain)
            if gain > 1e-5:
                assert int(z[f'{arch}_c{c}_interval_better']) == 1
            for k in range(1, L + 1):
                l, u = gl[k][i].cpu(), gu[k][i].cpu()
                want = torch.where((l >= 0) & (u >= 0), 1, torch.where((l <= 0) & (u <= 0), 0, -1)).to(torch.int8)
                assert torch.equal(masks[k - 1][i].cpu(), want), ('mask', c, k)
            lay, idx, choice = z[f'{arch}_c{c}_decision'].tolist()
            assert int(masks[lay][i][idx]) == choice, ('mask of the split node', c)
        print(f'child_bounds {arch} B={B} math={sc.get_option("math")}: worst rel err {worst:.2e}, second passes {int(second.sum())}', flush=True)


def check_child_bounds_shapes(case):
    """gnnb_child_bounds on networks that are not the CIFAR ones (odd spatial sizes and channel counts, 5x5 / 3x3 / 4x4 kernels,
    stride 1 and 2, windows clipped at every border, three conv layers in a row) against the oracle, domain by domain."""
    from torch import nn
    from gnn_branching_b200 import Flatten, Scorer, netspec_from_modules
    from gnn_branching_b200.frontier import interval_root_bounds
    from oracle import kw_bounds_oracle as KW
    if case == 'odd_shapes':
        layers = [nn.Conv2d(2, 5, 3, stride=1, padding=1), nn.ReLU(), nn.Conv2d(5, 6, 3, stride=2, padding=1), nn.ReLU(),
                  Flatten(), nn.Linear(6 * 5 * 4, 37), nn.ReLU()]
        shape = (2, 9, 7)
    else:
        layers = [nn.Conv2d(1, 4, 5, stride=1, padding=2), nn.ReLU(), nn.Conv2d(4, 4, 3, stride=1, padding=1), nn.ReLU(),
                  nn.Conv2d(4, 3, 4, stride=2, padding=1), nn.ReLU(), Flatten(), nn.Linear(3 * 6 * 6, 150), nn.ReLU(),
                  nn.Linear(150, 9), nn.ReLU()]
        shape = (1, 12, 12)
    g = torch.Generator().manual_seed(5)
    for m in layers:
        for q in m.parameters():
            q.data = torch.randn(q.shape, generator=g) * (0.3 if q.dim() > 1 else 0.1)
    net = netspec_from_modules(layers, shape, name='custom')
    x = torch.randn(shape, generator=g).reshape(-1)
    wp, bp, eps = torch.randn(net.hidden_sizes[-1], generator=g) * 0.3, 0.1, 0.05
    lbs, ubs = KW.root_bounds(net, x, eps, wp, bp)
    L = net.L
    decs = []
    for lay in range(L):
        amb = ((lbs[lay + 1] < 0) & (ubs[lay + 1] > 0)).nonzero().view(-1)
        for choice in (0, 1):
            if amb.numel():
                decs.append((lay, int(amb[int(torch.randint(0, amb.numel(), (1,), generator=g))]), choice))
    B = len(decs)
    assert B >= 4
    sc = Scorer(0)
    sc.set_network(net, key=net.key)
    sc.set_option('math', int(os.environ.get('GNNB_TEST_MATH', '0')))
    dec = torch.tensor(decs, dtype=torch.int32)
    gl, gu, masks, second = sc.child_bounds(x.reshape(1, -1), eps, wp.reshape(1, -1).repeat(B, 1), torch.full((B,), bp),
                                            [t.reshape(1, -1).repeat(B, 1) for t in lbs], [t.reshape(1, -1).repeat(B, 1) for t in ubs],
                                            dec[:, 0], dec[:, 1], dec[:, 2])
    torch.cuda.synchronize()
    worst = 0.0
    for i, (lay, idx, choice) in enumerate(decs):
        ol, ou, _ = KW.child_bounds(net, x, eps, wp, bp, lbs, ubs, (lay, idx), choice)
        for k in range(L + 2):
            e = max(float((gl[k][i].cpu() - ol[k]).abs().max()), float((gu[k][i].cpu() - ou[k]).abs().max())) / max(1.0, float(ou[k].abs().max()))
            worst = max(worst, e)
            assert e <= 5e-5, (case, i, k, e)
    print(f'child_bounds {case}: {B} children, worst rel err {worst:.2e}', flush=True)


def check_frontier_step(arch):
    """FrontierStep (pick -> split -> gnnb_child_bounds -> gnnb_score -> add, device-resident) against the pieces it is made
    of: the first step's two children carry the oracle's child bounds of the root for the root's GNN decision; afterwards, over
    several batched steps, every child's lower bound is at least its parent's, the queue holds exactly the children that were
    kept, and its global lower bound never decreases."""
    import numpy as np
    from golden_io import GOLDEN
    from gnn_branching_b200 import FrontierStep
    from oracle import kw_bounds_oracle as KW
    net, lbs, ubs, wp, bp = load_root(arch)
    x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))[f'{arch}_x'].copy()).reshape(-1)
    model = GraphNet(2, 64, math='tc')
    model.load_state_dict(load_gnn('random'))
    model = model.eval().cuda()
    fs = FrontierStep(model, net, x, 0.145, wp, bp, capacity=8192, decision_bound=float('inf'))
    fs.seed_root(lbs, ubs)
    assert len(fs.queue) == 1
    root = fs.queue.pick(1, float('inf'))
    dec = root.decision[0].tolist()
    fs.queue.add(root)
    st = fs.step(8)
    assert (st.picked, st.children, st.added, st.infeasible) == (1, 2, 2, 0) and len(fs.queue) == 2, st
    kids = fs.queue.pick(2, float('inf'))
    for i in range(2):
        # which side is this child?  the split node's bound is 0 on the fixed side
        side = 0 if float(kids.ub[dec[0] + 1][i, dec[1]]) == 0.0 else 1
        ol, ou, _ = KW.child_bounds(net, x, 0.145, wp, bp, lbs, ubs, dec, side)
        for k in range(net.L + 2):
            e = max(float((kids.lb[k][i].cpu() - ol[k]).abs().max()), float((kids.ub[k][i].cpu() - ou[k]).abs().max())) / max(1.0, float(ou[k].abs().max()))
            assert e <= 5e-5, ('child', i, k, e)
        assert float(kids.lower_bound[i]) == float(kids.lb[net.L + 1][i, 0])
        assert int(kids.mask[i, sum(net.hidden_sizes[:dec[0]]) + dec[1]]) == side
    assert {0 if float(kids.ub[dec[0] + 1][i, dec[1]]) == 0.0 else 1 for i in range(2)} == {0, 1}
    fs.queue.add(kids)
    glb, size = fs.queue.global_lb, 2
    dropped = 0
    for B in (2, 4, 8, 16, 32, 64, 128, 256):           # deep enough for splits that contradict each other (infeasible children)
        st = fs.step(B)
        size += st.added - st.picked
        dropped += st.infeasible
        assert st.children == 2 * st.picked and st.added <= st.children - st.infeasible and len(fs.queue) == size, (st, size)
        assert st.global_lb >= glb - 1e-6, (st.global_lb, glb)      # children are never looser than their parents
        glb = st.global_lb
    print(f'frontier_step {arch}: queue {len(fs.queue)} domains, {dropped} infeasible children dropped, global lb {glb:.4f}', flush=True)
    del fs
    # the threshold rule (relu_conv_gnnkwthreshold.py:145-203) with a threshold nothing passes: the KW decision is bounded for
    # every parent and wins exactly where its children improve the bound more.  First step against the oracles (BaBSR decision,
    # child bounds of both decisions, the improvement formula), then batched steps on invariants.
    from oracle import babsr_oracle as BO
    fs = FrontierStep(model, net, x, 0.145, wp, bp, capacity=8192, decision_bound=float('inf'), kw_fallback=True, branching_threshold=1e9)
    fs.seed_root(lbs, ubs)
    root = fs.queue.pick(1, float('inf'))
    gdec = root.decision[0].tolist()
    fs.queue.add(root)
    st = fs.step(1)
    assert st.kw_tried == 1 and st.added == 2, st
    L = net.L
    from gnn_branching_b200 import Frontier
    m_cpu = torch.cat([torch.where((lbs[k] < 0) & (ubs[k] > 0), 1.0, 0.0) for k in range(1, L + 1)]).reshape(1, -1)
    e = torch.empty(0)
    fr_cpu = Frontier(net=net, lb=[t.reshape(1, -1) for t in lbs], ub=[t.reshape(1, -1) for t in ubs], dual=[], prim_pre=[], prim_post=[],
                      prim_out=e, primal_input=e, Wp=wp.reshape(1, -1), bp=torch.tensor([bp]), mask=m_cpu)
    sc_, ic_ = BO.babsr_scores(fr_cpu)
    kdec = BO.babsr_decide(sc_, ic_, m_cpu, net.hidden_sizes, [0], [0] + list(range(1, L)), 0)[0][0]
    kdec = [int(kdec[0]), int(kdec[1])]

    def improvement(dec):
        lows = []
        for side in (0, 1):
            ol, ou, _ = KW.child_bounds(net, x, 0.145, wp, bp, lbs, ubs, dec, side)
            lows.append(min(float(ol[L + 1]), 0.0))
        plb = float(lbs[L + 1])
        return (lows[0] + lows[1] - 2 * plb) / (-2 * plb)
    gi, ki = improvement(gdec), improvement(kdec)
    want = kdec if (kdec != gdec and ki > gi) else gdec
    assert st.kw_used == int(want == kdec and kdec != gdec), (st, gdec, kdec, gi, ki)
    kids = fs.queue.pick(2, float('inf'))
    sides = {0 if float(kids.ub[want[0] + 1][i, want[1]]) == 0.0 else (1 if float(kids.lb[want[0] + 1][i, want[1]]) == 0.0 else -1) for i in range(2)}
    assert sides == {0, 1}, ('the children are not the two sides of the winning decision', want, gdec, kdec)
    fs.queue.add(kids)
    glb, size, tried, used = fs.queue.global_lb, 2, 0, 0
    for B in (2, 4, 8, 16, 32, 64):
        st = fs.step(B)
        size += st.added - st.picked
        tried += st.kw_tried; used += st.kw_used
        assert st.kw_tried == st.picked and st.kw_used <= st.kw_tried and len(fs.queue) == size, (st, size)
        assert st.global_lb >= glb - 1e-6
        glb = st.global_lb
    print(f'frontier_step {arch} with the KW threshold rule: root gnn {gdec} ({gi:.4f}) kw {kdec} ({ki:.4f}); {used} of {tried} parents took the KW decision', flush=True)


if __name__ == '__main__':
    {'frontier_step': check_frontier_step, 'kw_bounds': check_kw_bounds, 'fused': check_fused,
     'child_bounds': check_child_bounds, 'child_bounds_shapes': check_child_bounds_shapes}[sys.argv[1]](sys.argv[2])
    print('ok')
