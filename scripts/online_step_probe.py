"""Cost of online fine-tuning inside the frontier step: FrontierStep(kw_fallback=True) with online off and on, alternating,
on base and deep from the seeded root (tests/golden), up to --max-b parents per step, --steps steps per run.

Reports per run: children/s over the timed steps, and for online runs the parents trained on (m), the gradient pass
(gnnb_score_grad_device, host clock around a synchronised call) in ms per step and per wave, and the wave size.  The card's
name and power limit are read in the same process.

Usage: python scripts/online_step_probe.py [--steps 14] [--max-b 512] [--reps 2] [--out FILE]"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np                                               # noqa: E402
import torch                                                     # noqa: E402

from golden_io import GOLDEN, load_gnn, load_root                # noqa: E402
from gnn_branching_b200 import FrontierStep, GraphNet            # noqa: E402


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or f'{torch.cuda.get_device_name(0)} (power limit not readable)'


def run(arch, online, steps, max_b):
    net, lbs, ubs, wp, bp = load_root(arch)
    x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))[f'{arch}_x'].copy()).reshape(-1)
    model = GraphNet(2, 64, math='tc')
    model.load_state_dict(load_gnn('random'))
    model = model.eval().cuda()
    fs = FrontierStep(model, net, x, 0.145, wp, bp, capacity=1 << 16, decision_bound=float('inf'), kw_fallback=True, online=online)
    fs.seed_root(lbs, ubs)
    grad = []                                      # (ms, m, waves) per gradient pass
    sc = fs.scorer
    inner = sc.score_grad

    def timed(fr, terms):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = inner(fr, terms)
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0)
        w = sc.get_option('grad_workspace_domains')
        m = int((terms[0] >= 0).sum()) // 2
        grad.append((ms, m, -(-m // w) if w else 0, w))
        return out
    sc.score_grad = timed
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    children = trained = 0
    for _ in range(steps):
        st = fs.step(max_b)
        children += st.children
        trained += st.online_trained
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dict(children=children, s=dt, trained=trained, grad=grad, queue=len(fs.queue))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=14)
    ap.add_argument('--max-b', type=int, default=512)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('online_step_probe needs a CUDA device')
    lines = [f'card: {card()}', f'steps {a.steps}, up to {a.max_b} parents per step, kw_fallback=True, branching_threshold 0.2, '
             'random GNN weights; times: host clock around synchronised work']
    for arch in ('base', 'deep'):
        run(arch, True, 2, 8)                       # warm-up: modules, workspaces, the gradient arena
        for rep in range(a.reps):
            for online in (False, True):
                r = run(arch, online, a.steps, a.max_b)
                line = (f'{arch} rep {rep} online={int(online)}: {r["children"]} children in {r["s"]:.3f} s = '
                        f'{r["children"] / r["s"]:.0f} children/s, queue {r["queue"]}')
                if online:
                    g = r['grad']
                    ms = sum(x[0] for x in g)
                    waves = sum(x[2] for x in g)
                    line += (f'; {len(g)} gradient passes, {r["trained"]} parents trained on, gradient pass {ms:.1f} ms '
                             f'({ms / max(len(g), 1):.1f} ms per pass, {ms / max(waves, 1):.1f} ms per wave, '
                             f'{ms / 1e3 / r["s"] * 100:.0f}% of the run), wave size {max((x[3] for x in g), default=0)}')
                    line += '\n    per pass (ms, m, waves): ' + ' '.join(f'({x[0]:.1f}, {x[1]}, {x[2]})' for x in g)
                lines.append(line)
                print(line, flush=True)
    text = '\n'.join(lines) + '\n'
    print(lines[0])
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
