"""Cost of the top-k branching candidates and of strong branching on one GPU: python scripts/topk_probe.py [--out FILE] [--reps N]

(a) gnnb_score against gnnb_score_topk with k in {1, 4, 16, 64}: base x 1 024, wide x 4 096 and deep x 4 096 subdomains, DEVICE
    buffers and pinned HOST buffers; ms per call, median and min - max of --reps runs of 20 calls each, the variants alternating
    run by run.  A call ends in a device synchronise, so the time is the whole call.  A separate pass with option "profile" = 1
    reports the last launch of each wave alone (the argmax kernel for gnnb_score and k = 1, the top-k kernel otherwise).
(b) gnnb_topk alone over [1 024, n] random scores with a 60 % candidate mask, n in {3 172, 6 756, 100 000}, same timing.
(c) FrontierStep on base from the seeded root (decision bound 0), up to 512 parents per step, for strong_branching_k in
    {1, 2, 4, 8} and strong_branching_kw_k in {0, 2}: children per second over a fixed number of steps, and the queue's global lower bound and
    size after them.  The bounds are the KW / interval surrogate of the LP (bab_step.py), so are these lower bounds.
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from golden_io import GOLDEN, load_gnn, load_root  # noqa: E402
from gnn_branching_b200 import FrontierStep, GraphNet, Scorer, synthetic_frontier  # noqa: E402

KS = (1, 4, 16, 64)
STEPS = 14


def timed(variants, reps, calls=20):
    """{name: [ms per call of each run]}: the variants alternate run by run."""
    for fn in variants.values():       # warm-up: workspace, result buffers, modules
        fn()
        fn()
    torch.cuda.synchronize()
    runs = {k: [] for k in variants}
    for _ in range(reps):
        for name, fn in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(calls):
                fn()
            torch.cuda.synchronize()
            runs[name].append((time.perf_counter() - t0) / calls * 1e3)
    return runs


def cell(v):
    return f'{statistics.median(v):8.3f} ({min(v):.3f}-{max(v):.3f})'


def scoring(out, reps):
    sd = load_gnn('random')
    out('(a) gnnb_score vs gnnb_score_topk, random GNN weights, ms per call: median (min-max) of '
        f'{reps} runs x 20 calls; "+%" = median over gnnb_score')
    out(f'{"case":>18} {"variant":>10} {"ms":>26} {"+%":>7}')
    for arch, B in (('base', 1024), ('wide', 4096), ('deep', 4096)):
        net, lbs, ubs, wp, bp = load_root(arch)
        fr_dev = synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=2000, device='cuda')
        sc = Scorer(0)
        sc.set_gnn(sd)
        sc.set_network(net, key=net.key)
        for mem in ('device', 'host'):
            fr = fr_dev if mem == 'device' else fr_dev.cpu().pin()
            variants = {'score': lambda: sc.score(fr, return_scores=False, check=False)}
            for k in KS:
                variants[f'topk{k}'] = (lambda k=k: sc.score_topk(fr, k, check=False))
            runs = timed(variants, reps)
            base = statistics.median(runs['score'])
            for name, v in runs.items():
                rel = 100.0 * (statistics.median(v) / base - 1.0)
                out(f'{f"{arch} x {B} {mem}":>18} {name:>10} {cell(v):>26} {rel:>+7.2f}')
        # the last launch of every wave on its own (option "profile"; events around each stage launch)
        sc.set_option('profile', 1)
        parts = []
        for name, fn in [('argmax', lambda: sc.score(fr_dev, return_scores=False, check=False))] + \
                [(f'topk{k}', (lambda k=k: sc.score_topk(fr_dev, k, check=False))) for k in KS]:
            fn()
            sc.profile_reset()
            for _ in range(20):
                fn()
            torch.cuda.synchronize()
            p = sc.profile_read()
            total = sum(v['ms'] for v in p.values())
            parts.append(f'{name} {p["argmax"]["ms"] / p["argmax"]["launches"] * 1e3:.1f} us '
                         f'({100.0 * p["argmax"]["ms"] / total:.2f} % of the staged kernel time)')
        sc.set_option('profile', 0)
        out(f'{f"{arch} x {B}":>18} last launch per wave, device, profile = 1: ' + '; '.join(parts))


def topk_alone(out, reps):
    out('')
    out(f'(b) gnnb_topk alone, B = 1 024, random scores, 60 % candidates; ms per call: median (min-max) of {reps} runs x 20 calls')
    sc = Scorer(0)
    g = torch.Generator(device='cuda').manual_seed(5)
    for n in (3172, 6756, 100000):
        s = torch.randn(1024, n, generator=g, device='cuda')
        m = (torch.rand(1024, n, generator=g, device='cuda') < 0.6).float()
        runs = timed({f'k={k}': (lambda k=k: sc.topk(s, k, mask=m)) for k in KS}, reps)
        out(f'  n = {n:>6}: ' + '; '.join(f'{name} {cell(v).strip()}' for name, v in runs.items()))


def strong(out):
    out('')
    out(f'(c) FrontierStep, base, seeded root, decision bound 0, up to 512 parents per step, {STEPS} steps, random GNN weights, '
        'tensor cores; lower bounds are the KW / interval surrogate LP bounds')
    out(f'{"k":>3} {"kw_k":>5} {"children":>9} {"s":>7} {"children/s":>11} {"extra pairs":>12} {"changed":>8} '
        f'{"global lb (surrogate LP)":>24} {"queue":>7}')
    net, lbs, ubs, wp, bp = load_root('base')
    x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))['base_x'].copy()).reshape(-1)
    model = GraphNet(2, 64)
    model.load_state_dict(load_gnn('random'))
    model = model.eval().cuda()
    for kw_k in (0, 2):
        for k in (1, 2, 4, 8):
            fs = FrontierStep(model, net, x, 0.145, wp, bp, capacity=1 << 16,
                              strong_branching_k=k, strong_branching_kw_k=kw_k)
            fs.seed_root(lbs, ubs)
            torch.cuda.synchronize()
            children = bounded = changed = 0
            t0 = time.perf_counter()
            for _ in range(STEPS):
                st = fs.step(512)
                children += st.children
                bounded += st.sb_bounded
                changed += st.sb_changed
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            glb = fs.queue.global_lb if len(fs.queue) else float('nan')
            out(f'{k:>3} {kw_k:>5} {children:>9} {dt:>7.2f} {children / dt:>11.0f} {bounded:>12} {changed:>8} '
                f'{glb:>24.5f} {len(fs.queue):>7}')
            del fs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='also write the report to this file')
    ap.add_argument('--reps', type=int, default=7)
    a = ap.parse_args()
    lines = []

    def out(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    out(f'GPU 0: {q.stdout.strip() or torch.cuda.get_device_name(0)} (name, power limit, max SM clock); torch {torch.__version__}')
    scoring(out, a.reps)
    topk_alone(out, a.reps)
    strong(out)
    if a.out:
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
