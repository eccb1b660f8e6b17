"""Cost and range sweep of option "rescore" on one GPU: python scripts/rescore_probe.py [--out FILE] [--reps N]

Cost: a base x 1 024 DEVICE frontier with 0, 1, 8 and 64 subdomains pushed out of the tensor-core operand range (their duals
scaled until the option-off call reports NaN); ms per call with the option off and on, alternating, over --reps runs of 20
calls each (median and min - max of the runs).  A call ends in a device synchronise, so the time is the whole call.

Range sweep, base / wide / deep x 1 024 subdomains, random GNN weights unless stated: bounds (lb, ub of every layer) x {0.01,
100}, duals x {1e-3, 1e3, 1e6}, GNN weight matrices x {0.25, 4} (biases unchanged), and the shipped checkpoint.  Per case: the
largest per-subdomain max|s - s_oracle| / max|s_oracle| over candidate rows of a 12-subdomain slice (option on), whether the
option-off call reported NaN, and how many subdomains the option-on call re-scored.
"""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch  # noqa: E402

from golden_io import ARCHS, load_gnn, load_root  # noqa: E402
from gnn_branching_b200 import Scorer, synthetic_frontier, _lib  # noqa: E402
from oracle import graphnet_oracle as O  # noqa: E402

B = 1024


def scorer(sd, net, rescore):
    sc = Scorer(0, rescore=rescore)
    sc.set_gnn(sd)
    sc.set_network(net, key=net.key)
    return sc


def nan_reported(sc):
    n = C.c_int64(0)
    return sc.lib.gnnb_check(sc.h, C.c_void_p(torch.cuda.current_stream().cuda_stream), C.byref(n)) == _lib.GNNB_ERR_NAN


def frontier(arch, seed):
    net, lbs, ubs, wp, bp = load_root(arch)
    return net, synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=seed, device='cuda')


def with_duals(fr, rows, factor):
    fr = fr._map(lambda t: t.clone())
    for d in fr.dual:
        d[rows] *= factor
    return fr


def cost(out, reps):
    sd = load_gnn('random')
    net, fr = frontier('base', 2000)
    off, on = scorer(sd, net, False), scorer(sd, net, True)
    # the factor: the smallest power of ten at which one scaled subdomain overflows the tensor-core pass
    factor = None
    for e in range(4, 12):
        off.score(with_duals(fr, [0], 10.0 ** e), check=False)
        if nan_reported(off):
            factor = 10.0 ** e
            break
    out(f'cost: base x {B}, DEVICE, random weights, duals of the overflow subdomains x {factor:g}; {reps} runs x 20 calls per cell')
    out(f'{"overflowing":>12} {"off ms":>10} {"(min-max)":>16} {"on ms":>10} {"(min-max)":>16} {"rescored":>9}')
    g = torch.Generator().manual_seed(7)
    for k in (0, 1, 8, 64):
        rows = sorted(torch.randperm(B, generator=g)[:k].tolist())
        f = with_duals(fr, rows, factor) if k else fr
        runs = {False: [], True: []}
        for sc in (off, on):              # warm-up
            sc.score(f, check=False)
            nan_reported(sc)
        for _ in range(reps):
            for resc, sc in ((False, off), (True, on)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(20):
                    sc.score(f, check=False)
                torch.cuda.synchronize()
                runs[resc].append((time.perf_counter() - t0) / 20 * 1e3)
                nan_reported(sc)
        m = {r: statistics.median(v) for r, v in runs.items()}
        out(f'{k:>12} {m[False]:>10.3f} {f"({min(runs[False]):.3f}-{max(runs[False]):.3f})":>16} {m[True]:>10.3f} '
            f'{f"({min(runs[True]):.3f}-{max(runs[True]):.3f})":>16} {on.rescored:>9}')


def sweep(out):
    out(f'range sweep: {B} subdomains per case; error = max over a 12-subdomain slice of max|s - s_oracle| / max|s_oracle| '
        '(candidate rows, option on)')
    out(f'{"arch":>5} {"case":>18} {"error":>10} {"NaN off":>8} {"rescored":>9}')
    ids = sorted({0, 1, B // 7, B // 3, B // 2 - 1, B // 2, (2 * B) // 3, B - 130, B - 129, B - 3, B - 2, B - 1})
    for arch in ARCHS:
        net, base = frontier(arch, 1000 * (2 + ARCHS.index(arch)))
        cases = []
        for f in (0.01, 100.0):
            cases.append((f'bounds x {f:g}', 'random', base._map(lambda t: t.clone())))
            cases[-1][2].lb[:] = [t * f for t in base.lb]
            cases[-1][2].ub[:] = [t * f for t in base.ub]
        for f in (1e-3, 1e3, 1e6):
            cases.append((f'duals x {f:g}', 'random', with_duals(base, list(range(B)), f)))
        for f in (0.25, 4.0):
            cases.append((f'weights x {f:g}', f'random*{f:g}', base))
        cases.append(('shipped', 'shipped', base))
        for name, weights, fr in cases:
            if '*' in weights:
                f = float(weights.split('*')[1])
                sd = {k: (v * f if k.endswith('weight') else v) for k, v in load_gnn('random').items()}
            else:
                sd = load_gnn(weights)
            off, on = scorer(sd, net, False), scorer(sd, net, True)
            off.score(fr, return_scores=False, check=False)
            nan_off = nan_reported(off)
            _, idx, s = on.score(fr, check=False)
            nan_on = nan_reported(on)
            sl = fr._map(lambda t: t[ids]).cpu().contiguous()
            s_or, _ = O.gnn_forward(sd, sl)
            s = s[ids].cpu()
            err = 0.0
            for j in range(len(ids)):
                m = sl.mask[j] != 0
                if not bool(m.any()):
                    continue
                d = float((s[j][m].double() - s_or[j][m].double()).abs().max()) / max(float(s_or[j][m].abs().max()), 1e-30)
                err = max(err, d) if d == d else float('nan')
            note = '  (NaN also in fp32)' if nan_on else ''
            out(f'{arch:>5} {name:>18} {err:>10.2e} {str(nan_off):>8} {on.rescored:>9}{note}')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='also write the report to this file')
    ap.add_argument('--reps', type=int, default=7)
    a = ap.parse_args()
    lines = []

    def out(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    out(f'GPU 0: {q.stdout.strip() or torch.cuda.get_device_name(0)} (name, power limit); torch {torch.__version__}')
    cost(out, a.reps)
    out('')
    sweep(out)
    if a.out:
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
