#!/usr/bin/env python
"""Benchmark of the GNN branching-score hot path: subdomains scored per second on a B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload base|wide|deep] [--domains B_per_gpu] [--dump-outputs DIR]
    python bench.py --impl reference ...      # the reference algorithm on the host CPU (oracle port)

One step = one pass of the hot path over one frontier of synthetic subdomains (SURVEY §8d generator):
at N = 1 the workload is BASELINE.json configs[1], cifar_base_kw x 1 024 subdomains; at N > 1 every rank scores
the same number of subdomains (weak scaling, no data-path collective) and the per-subdomain winners are
all-gathered with NCCL inside the timed region.  Prints ONE JSON line (rank 0).  The frontiers are seeded, so two runs
with the same arguments score the same inputs: --dump-outputs lets two builds be compared winner for winner.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

METRIC = 'gnn_subdomains_scored_per_sec'
UNIT = 'subdomains/s'
DEFAULT_DOMAINS = {'base': 1024, 'wide': 4096, 'deep': 4096}
CPU_SAMPLE = 32          # subdomains per CPU-baseline pass (the reference's CPU rate is flat from B = 4, SURVEY §6.3)
FRONTIER_TOTAL = 65536   # BASELINE configs[4]: the base frontier sharded over N > 1 GPUs


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='base', choices=['base', 'wide', 'deep'])
    ap.add_argument('--domains', type=int, default=0, help='subdomains per GPU per step (default: BASELINE config size)')
    ap.add_argument('--math', default=None, choices=['tc', 'simt'])
    ap.add_argument('--chunk', type=int, default=0)
    ap.add_argument('--weights', default='random', choices=['random', 'shipped'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-babsr', action='store_true')
    ap.add_argument('--no-online', action='store_true')
    ap.add_argument('--no-queue', action='store_true')
    ap.add_argument('--no-step', action='store_true', help='skip the device-resident branch-and-bound step (pick, bound, score, add)')
    ap.add_argument('--no-secondary', action='store_true', help='skip the wide / deep x 4096 secondary objects of the default line')
    ap.add_argument('--opt', action='append', default=[], help='library option key=value (e.g. fuse=0, prop_share=40)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the winners of the last timed step (what the caller receives) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    return args


def load_problem(workload):
    """Verified net + KW root bounds of one property (tests/golden/nets.npz) and the GNN weights."""
    from golden_io import load_root
    return load_root(workload)


def load_weights(which):
    from golden_io import load_gnn
    return load_gnn(which)


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / throttle reasons of one GPU sampled DURING the timed region: NVML (nvidia_ml_py) polled every 5 ms from a
    thread — a 50 ms timed region still gets ~10 samples — with `nvidia-smi -lms 50` as the fallback."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    BITS = {'sw_power_cap': 0x4, 'hw_slowdown': 0x8, 'sw_thermal_slowdown': 0x20, 'hw_thermal_slowdown': 0x40}

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nv, self.h, self.stop = index, [], None, None, None, False
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + uuid) if not uuid.startswith('GPU-') else uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    pw = 0.0
                self.samples.append((sm, mask, pw))
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        self.samples = []
        if self.nv is not None:
            self.stop = False
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return self
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '50', '-i', str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def __exit__(self, *a):
        if self.nv is not None:
            self.stop = True
            self.t.join(timeout=2)
        elif self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            self.t.join(timeout=2)

    def count(self):
        return len(self.samples) if self.nv is not None else len(self.rows)

    def summary(self):
        if self.nv is not None and self.samples:
            sm = [q[0] for q in self.samples]
            reasons = sorted(n for n, bit in self.BITS.items() if any(q[1] & bit for q in self.samples))
            return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': self.max_mhz, 'reasons': reasons,
                    'power_w_max': max(q[2] for q in self.samples), 'samples': len(sm),
                    'source': 'nvml polled every 5 ms over the timed region (+ identical untimed steps until 8 samples)'}
        sm, mx, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': max(mx), 'reasons': sorted(reasons),
                'power_w_max': max(power), 'samples': len(sm), 'source': 'nvidia-smi -lms 50'}


def run_timed(step, local_step, K, barrier, record0, record1, clock_samples, sync, min_samples=8, max_extra=400):
    """The timed region: barrier, K steps between the two event records, barrier.  `step` may contain collectives (every
    rank calls it exactly K times); afterwards the identical load is kept running with `local_step` — rank-LOCAL work only,
    because every rank runs a different number of these — until the clock sampler has `min_samples` samples under load
    (a K x 5 ms region can end before NVML has answered a handful of times).  What the last timed step returned is kept in
    `run_timed.last`."""
    barrier()
    record0()
    for i in range(K):
        out = step(i)
    record1()
    run_timed.last = out
    barrier()
    extra = 0
    while clock_samples() < min_samples and extra < max_extra:
        local_step(extra)
        extra += 1
        if extra % 4 == 0:
            sync()
    sync()
    run_timed.extra = extra
    return extra


run_timed.extra = 0
run_timed.last = None


def _run_ref_runner(device, workload, weights, batches, reps, warmup=1, timeout=900):
    """oracle/ref_runner.py in its own process (CPU runs must not see a GPU; SURVEY §8d).  Returns its JSON or None."""
    from oracle import ref_runner
    if not ref_runner.available():
        return None
    env = dict(os.environ)
    if device == 'cpu':
        env['CUDA_VISIBLE_DEVICES'] = ''
    for k in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE', 'MASTER_ADDR', 'MASTER_PORT'):
        env.pop(k, None)
    cmd = [sys.executable, os.path.join(ROOT, 'oracle', 'ref_runner.py'), '--device', device, '--workload', workload, '--weights', weights,
           '--batches', ','.join(str(b) for b in batches), '--reps', str(reps), '--warmup', str(warmup)]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        if r.returncode != 0:
            return {'error': (r.stderr or r.stdout)[-300:]}
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:          # a baseline must never take the bench line down
        return {'error': repr(e)[:300]}


def cpu_baseline(workload, weights, threads=None, reps=3, warmup=1):
    """The reference GNN forward on the host cores: the UNMODIFIED graphnet/graph_conv.py staged in oracle/_ref (kind
    "reference") when it is there, else the oracle port (kind "port").  B = 1 latency (the reference's native usage) and the
    best rate over B in {1, 8, 32} (its CPU rate is flat from B = 4, SURVEY §6.3)."""
    threads = threads or os.cpu_count()
    ref = _run_ref_runner('cpu', workload, weights, (1, 8, CPU_SAMPLE), reps, warmup)
    if ref and 'error' not in ref:
        pb = ref['per_batch']
        times = pb[str(CPU_SAMPLE)]['times_s']
        return {'value': ref['value'], 'unit': UNIT, 'cores': ref['cores'], 'kind': 'reference', 'best_batch': ref['best_batch'],
                'b1_latency_ms': ref['b1_latency_ms'], 'rate_by_batch': {k: v['rate'] for k, v in pb.items()},
                'sample': f'unmodified graphnet/graph_conv.py GraphNet.forward (oracle/_ref, own process without a GPU), cifar_{workload}_kw, '
                          f'B in (1, 8, {CPU_SAMPLE}) x {reps} passes each, best pass of the best batch size'}, times
    import torch
    from gnn_branching_b200 import synthetic_frontier
    from oracle import graphnet_oracle as O
    torch.set_num_threads(threads)
    net, lbs, ubs, wp, bp = load_problem(workload)
    fr = synthetic_frontier(net, lbs, ubs, wp, bp, CPU_SAMPLE, seed=99)
    sd = load_weights(weights)
    with torch.no_grad():
        O.gnn_forward(sd, fr.slice(0, 4))                  # warm-up
        times = []
        for _ in range(reps):
            t0 = time.perf_counter()
            s, _ = O.gnn_forward(sd, fr)
            O.decide(s, fr.mask, net.hidden_sizes)
            times.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        O.gnn_forward(sd, fr.slice(0, 1))
        lat1 = time.perf_counter() - t0
    best = min(times)
    return {'value': CPU_SAMPLE / best, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'b1_latency_ms': lat1 * 1e3,
            'sample': f'{CPU_SAMPLE} cifar_{workload}_kw subdomains x {reps} passes, best pass; oracle/graphnet_oracle.py (fp32 torch-CPU '
                      f'restatement of graphnet/graph_conv.py) because oracle/_ref is not staged' + (f' ({ref["error"]})' if ref else ''),
            'median_value': CPU_SAMPLE / statistics.median(times)}, times


def run_reference(args):
    """--impl reference: the reference's own GNN forward (oracle/_ref, unmodified; else the oracle port) on this box's host
    cores, every step one pass over a CPU_SAMPLE-subdomain sample of the workload."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cb, times = cpu_baseline(args.workload, args.weights, reps=max(1, args.steps), warmup=max(1, args.warmup))
    per = sum(times) / len(times)
    # the same config keys as the B200 arm's line (the workload the rate stands for), with the bounded sample that was actually
    # timed stated beside it: the CPU rate per subdomain is flat in the batch size from B = 4 on (SURVEY §6.3)
    world = max(1, args.gpus)
    strong = world > 1 and not args.domains and args.workload == 'base'
    B = args.domains or (FRONTIER_TOTAL // world if strong else DEFAULT_DOMAINS[args.workload])
    wl_name = (f'cifar_base_kw frontier of {B * world} synthetic subdomains sharded across {world} GPUs ({B} per GPU per step)' if strong
               else f'cifar_{args.workload}_kw x {B} synthetic subdomains per GPU per step')
    line = {'impl': 'reference', 'metric': METRIC, 'value': CPU_SAMPLE / per, 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': len(times), 'warmup': args.warmup, 'ms_per_step': per * 1e3, 'higher_is_better': True,
            'scaling': 'strong' if strong else 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': wl_name, 'gnn': 'GraphNet(T=2,p=64)', 'weights': args.weights,
                       'sample': f'{CPU_SAMPLE}-subdomain sample of that workload per step, host CPU only (rank 0)'},
            'cpu_baseline': {**cb, 'value': CPU_SAMPLE / per},
            'e2e': {'value': CPU_SAMPLE / per, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


def kernel_rooflines(net, fr, prof, n_domains, T, peak_tf, peak_gbs, p=64):
    """Per-kernel-class algorithmic FLOPs / HBM bytes (DESIGN.md §4) against the live CUDA-event times.

    Bytes are the compulsory ones of the private layout: 256 B per node for every mu / nb row read or written once,
    relax' only for ambiguous rows (fraction taken from the frontier's bounds), the caller's inputs once."""
    import torch
    n = net.hidden_sizes
    L = len(n)
    mac = [a.macs_per_channel for a in net.affine]
    amb = [float(((fr.lb[k + 1] < 0) & (fr.ub[k + 1] > 0)).float().mean()) for k in range(L)]
    row = 4 * p                                                        # bytes of one embedding row (fp32 or fp16 hi + lo)
    flop, byts = {}, {}
    upd_f = 2 * 6 * p * p
    flop['update'] = sum(n) * (T * upd_f + (T - 1) * upd_f + (upd_f + 2 * (p * p + p)))
    byts['update'] = 2 * T * sum(nk * (2 * row + 8 + row * a) for nk, a in zip(n, amb)) + 4 * sum(n)
    flop['prop'] = 2 * p * (T * (sum(mac) + 0) + T * (sum(mac[1:]) + n[-1]) + (T - 1) * mac[0])
    n_all = [net.n0] + n
    fwd_rows = sum(n_all[k] + n_all[k + 1] for k in range(L))
    bwd_rows = sum(n_all[k + 1] + n_all[k] for k in range(1, L)) + n[-1]
    byts['prop'] = row * (T * fwd_rows + T * bwd_rows + (T - 1) * (n_all[1] + n_all[0]))
    flop['relax'] = sum(nk * a for nk, a in zip(n, amb)) * 2 * (14 * p + 7 * p * p)
    byts['relax'] = sum(nk * (8 + a * (28 + 2 * row)) for nk, a in zip(n, amb))
    flop['input'] = net.n0 * 2 * ((3 * p + p * p) + (T - 1) * (2 * p + 4 * p * p))
    byts['input'] = net.n0 * ((12 + row) + (T - 1) * (8 + 2 * row))
    groups = {'update': ['update_fwd', 'update_bwd', 'update_bwd_score'], 'prop': ['prop_fwd', 'prop_bwd'],
              'relax': ['relax'], 'input': ['input_embed', 'input_update'],
              'layer': ['layer_fwd', 'layer_bwd', 'layer_bwd_score']}
    fused_ms = sum(prof[m]['ms'] for m in groups['layer'] if m in prof)
    if fused_ms > 0:
        # fused launches (propagation + update of a layer): everything except the property layer's back-propagation and the
        # input-layer propagation; their nb hand-off goes through L2 and is not compulsory HBM traffic
        node_bytes = [nk * (row + 8 + row * am) for nk, am in zip(n, amb)]          # mu written + l, u + relax' per sweep
        fwd = sum(n_all[k] * row + node_bytes[k] for k in range(L))                # layer k+1 gathers layer k
        bwd = sum(n_all[k + 2] * row + node_bytes[k] for k in range(L - 1))        # layer k+1 gathers layer k+2
        byts['layer'] = T * (fwd + bwd) + 4 * sum(n[:-1])
        flop['layer'] = flop['update'] + flop['prop'] - 2 * p * (T - 1) * mac[0] - n[-1] * (T * upd_f + 2 * (p * p + p))
        flop['update'] = n[-1] * (T * upd_f + 2 * (p * p + p))                     # last hidden layer, backward sweeps
        byts['update'] = T * (n[-1] * row + node_bytes[-1]) + 4 * n[-1]
        flop['prop'] = 2 * p * (T - 1) * mac[0]                                    # input-layer propagation + property rank-1
        byts['prop'] = row * (T * n[-1] + (T - 1) * (n_all[1] + n_all[0]))
    names = {'layer': 'k_tc_fused (propagation gather-GEMM -> tensor memory -> node update chain of one layer, one kernel)',
             'update': 'k_tc_update (node update MLP chain, forward / backward / + score head)',
             'prop': 'k_tc_prop (embedding propagation through the verified network, gather-GEMM)',
             'relax': 'k_tc_relax (+ ambiguous-row compaction)', 'input': 'k_tc_input_embed / k_tc_input_update'}
    total_ms = sum(v['ms'] for v in prof.values()) or 1.0
    classes = {}
    for gname, members in groups.items():
        ms = sum(prof[m]['ms'] for m in members if m in prof)
        launches = sum(prof[m]['launches'] for m in members if m in prof)
        if ms <= 0:
            continue
        gbs = byts[gname] * n_domains / (ms * 1e-3) / 1e9
        tfs = flop[gname] * n_domains / (ms * 1e-3) / 1e12
        classes[gname] = {'ms': round(ms, 3), 'share_of_step': round(ms / total_ms, 4), 'launches': launches,
                          'avg_launch_ms': ms / max(launches, 1), 'hbm_gbs': gbs, 'hbm_frac': gbs / peak_gbs,
                          'tflops': tfs, 'tensor_frac': tfs / peak_tf,
                          'algorithmic_bytes_per_subdomain': byts[gname], 'algorithmic_flop_per_subdomain': flop[gname]}
    top = max(classes, key=lambda k: classes[k]['ms'])
    c = classes[top]
    # which roof is the nearer one: every product costs three fp16 MMA passes (fp32 accuracy), so the tensor pipe is 3 x as busy as
    # the algorithmic FLOPs say; the fused layer kernel sits closer to that roof than to the HBM one (ncu: tensor pipe 58 % active,
    # DRAM 42 %), the stand-alone kernels of the two-launch path closer to HBM
    hbm = {'achieved': c['hbm_gbs'], 'peak': peak_gbs, 'unit': 'GB/s', 'frac': c['hbm_frac'],
           'algorithmic_bytes_per_subdomain': c['algorithmic_bytes_per_subdomain']}
    tensor = {'achieved': c['tflops'], 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': c['tensor_frac'], 'frac_of_3_pass_ceiling': 3 * c['tensor_frac'],
              'algorithmic_flop_per_subdomain': c['algorithmic_flop_per_subdomain']}
    head = dict(tensor, bound='tensor') if 3 * c['tensor_frac'] >= c['hbm_frac'] else dict(hbm, bound='hbm')
    return {'bound': head['bound'], 'kernel': names[top], 'kernel_class': top, 'achieved': head['achieved'], 'peak': head['peak'],
            'unit': head['unit'], 'frac': head['frac'], 'launches': c['launches'], 'avg_launch_ms': c['avg_launch_ms'],
            'share_of_step': c['share_of_step'], 'tensor': tensor, 'hbm': hbm,
            'classes': classes, 'ambiguous_fraction': [round(a, 3) for a in amb],
            'kernel_ms': {k: round(v['ms'], 3) for k, v in prof.items()},
            '_bytes_per_subdomain': sum(byts.values())}


def measure_device(scorer, fronts, B, K, W, world, dev, local, gather):
    """Device-resident rate of one workload: W warm-up steps, K timed steps between CUDA events (barrier + synchronize on both
    sides, max over ranks), clocks sampled during the timed region, then a second pass of K steps with events around every
    launch for the per-kernel-class times."""
    import torch
    import torch.distributed as dist

    def score(fr):
        scorer.set_network(fr.net, key=fr.net.key)
        return scorer.score(fr, return_scores=False, check=False)

    rec = torch.empty(B, 2, dtype=torch.int32, device=dev) if world > 1 else None

    def step(i):
        fr = fronts[i % len(fronts)]
        if world > 1:      # the argmax kernel writes the packed (score, index) records the all-gather sends (SURVEY 8e)
            scorer.set_network(fr.net, key=fr.net.key)
            return gather(scorer.score_winners(fr, out=rec), B * world)
        best, idx, _ = score(fr)
        return best, idx

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(W):
        step(i)
    scorer.check()
    barrier()
    launches0 = scorer.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        run_timed(step, lambda i: score(fronts[i % len(fronts)]), K, barrier, ev0.record, ev1.record, clk.count, torch.cuda.synchronize)
        launches = (scorer.launches - launches0) * K // (K + run_timed.extra)      # every step issues the same launches
    scorer.check()
    outputs = tuple(t.clone() for t in run_timed.last)          # the gather writes a persistent buffer the passes below reuse
    ms = ev0.elapsed_time(ev1)
    # per-kernel-class durations: a second pass of K identical steps with CUDA events around every launch (on the launching
    # stream).  The events serialise consecutive launches (no programmatic overlap of a kernel's prologue with its
    # predecessor's tail), so the headline `value` above is measured without them
    scorer.set_option('profile', 1)
    scorer.profile_reset()
    for i in range(K):
        step(i)
    scorer.check()
    prof = scorer.profile_read()
    scorer.set_option('profile', 0)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return {'value': B * world * K / (ms * 1e-3), 'ms': ms, 'launches': launches, 'prof': prof, 'clocks': clk.summary(),
            'outputs': outputs}


DUMP_LIMIT = 64 * 10 ** 6      # bytes written by --dump-outputs


def dump_outputs(out_dir, best, idx):
    """The winners of the last timed step as DIR/best_score.npy (float32) and DIR/best_index.npy (float64: flat index of the
    chosen ReLU over all hidden layers, -1 where a subdomain has no candidate).  Past DUMP_LIMIT bytes, a fixed seeded sample
    of subdomains is written, their positions in DIR/sample_rows.npy."""
    import numpy as np
    best, idx = best.cpu().numpy().astype(np.float32), idx.cpu().numpy().astype(np.float64)
    n, headers = best.shape[0], 4096          # 4096: room for the .npy headers
    arrays = {'best_score': best, 'best_index': idx}
    # 12 bytes per subdomain: a 65 536-subdomain frontier writes 0.8 MB, so only very large --domains x --gpus runs sample;
    # a sampled row costs 20 bytes (its position in sample_rows.npy included)
    if n * (4 + 8) + headers > DUMP_LIMIT:
        rows = np.sort(np.random.default_rng(0).choice(n, (DUMP_LIMIT - headers) // (4 + 8 + 8), replace=False))
        arrays = {'best_score': best[rows], 'best_index': idx[rows], 'sample_rows': rows.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def measure_e2e(model, host_fronts, B, K, W, world, dev, gather):
    """The same metric through the public API with pinned HOST buffers: host->device copies of every step's inputs and the
    device->host read of the winners are inside the timed region (wall clock between barriers, max over ranks)."""
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    scorer = model.scorer(dev.index)
    rec = torch.empty(B, 2, dtype=torch.int32, device=dev) if world > 1 else None

    def step(i):
        fr = host_fronts[i % len(host_fronts)]
        if world == 1:
            return model.score_frontier(fr, return_scores=False)
        # inputs staged host -> device inside the call, records stay on the GPU, all-gather, then the whole frontier's winners are
        # read back by every rank (the device -> host read of the step's result)
        best, idx = gather(scorer.score_winners(fr, out=rec), B * world)
        return best.cpu(), idx.cpu()

    for i in range(min(W, 2)):
        step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        step(i)
    barrier()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    return {'value': B * world * K / dt, 'unit': UNIT, 'h2d_bytes_per_step': host_fronts[0].input_bytes(),
            'd2h_bytes_per_step': B * world * 8 if world > 1 else B * 8,
            'api': 'GraphNet.score_frontier(pinned host Frontier)' if world == 1 else
                   'Scorer.score_winners(pinned host Frontier) + dist.gather_winner_records + read-back of all winners'}


def measure_frontier_step(model, workload, dev, world, parents=256, steps=4):
    """Secondary object: the device-resident branch-and-bound step (gnn_branching_b200/bab_step.py) — every rank grows its own
    queue from the root of the same property, then `steps` steps of `parents` parents (2 x parents children: bounds part of
    update_the_model, GNN decision, add) are timed by the wall clock around the calls, max over ranks; and gnnb_child_bounds
    alone on one such batch.  LP values are surrogates (no Gurobi): see bab_step.py."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from golden_io import GOLDEN
    from gnn_branching_b200 import FrontierStep
    net, lbs, ubs, wp, bp = load_problem(workload)
    x = torch.from_numpy(np.load(os.path.join(GOLDEN, 'nets.npz'))[f'{workload}_x'].copy()).reshape(-1)

    def sync_ranks(v):          # every rank reaches every collective, whatever happened to it in between: max over ranks
        if world == 1:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    fs, err = None, None
    try:
        fs = FrontierStep(model, net, x, 0.145, wp, bp, capacity=(steps + 4) * 2 * parents, decision_bound=float('inf'), device=dev.index)
        fs.seed_root(lbs, ubs)
        while len(fs.queue) < parents:
            fs.step(parents)
        fs.step(parents)                              # one warm step at the timed size
        torch.cuda.synchronize()
    except Exception as e:
        err = e
    failed = sync_ranks(0.0 if err is None else 1.0)   # doubles as the barrier in front of the timed region
    dt, second, launches, infeasible = float('inf'), 0, 0, 0
    if not failed:
        try:
            l0, t0 = fs.scorer.launches, time.perf_counter()
            for _ in range(steps):
                st = fs.step(parents)
                second += st.second_pass
                infeasible += st.infeasible
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            launches = fs.scorer.launches - l0
        except Exception as e:
            err = e
    dt = sync_ranks(dt)
    if err is not None or failed or dt == float('inf'):
        raise RuntimeError(f'frontier step failed on a rank: {err!r}')
    children = 2 * parents * steps
    # the bound producer alone, on the children of one more batch of parents
    par = fs.queue.pick(parents, float('inf'))
    rep = lambda t: t.repeat_interleave(2, dim=0)
    n2 = 2 * par.B
    args = (fs.x, fs.eps, fs.Wp.expand(n2, -1), fs.bp.expand(n2), [rep(t) for t in par.lb], [rep(t) for t in par.ub],
            rep(par.decision)[:, 0], rep(par.decision)[:, 1], torch.arange(n2, device=dev, dtype=torch.int32) & 1)
    fs.scorer.child_bounds(*args)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        fs.scorer.child_bounds(*args)
    torch.cuda.synchronize()
    cb_ms = (time.perf_counter() - t0) / 3 * 1e3
    # executed work of the bound producer.  Conv layers behind conv layers take the windowed recursion (k_kw_cone: per position
    # and output channel, the footprint windows of the layers in front); the other layers and the property output the dense
    # recursion: ceil(n_k / 64) groups of 64 columns, each pushed through A_j^T for every layer j < k as fp32 [n, 64] column blocks
    n = [net.n0] + net.hidden_sizes
    mac = [a.weight.numel() * (a.out_shape[1] * a.out_shape[2] if a.kind == 'conv' else 1) for a in net.affine]
    flop = byts = 0
    for k in list(range(2, net.L + 1)) + [net.L + 1]:
        cone = k <= net.L and all(a.kind == 'conv' for a in net.affine[:k])
        if cone:
            a_k = net.affine[k - 1]
            h = w = 1
            for j in range(k, 0, -1):                 # window of layer j - 1 under one position of layer k (unclipped)
                a_j = net.affine[j - 1]
                ks = a_j.weight.shape[2]
                taps = -(-ks // a_j.stride) ** 2 if j < k else 0
                if j < k:                             # A_j^T on the window: every element of window j - 1 x valid taps x C_j x columns
                    hh, ww = (h - 1) * a_j.stride + ks, (w - 1) * a_j.stride + ks
                    flop += a_k.out_shape[1] * a_k.out_shape[2] * 2 * a_k.out_shape[0] * a_j.in_shape[0] * hh * ww * taps * a_j.out_shape[0]
                h, w = (h - 1) * a_j.stride + ks, (w - 1) * a_j.stride + ks
            byts += 2 * 4 * n[k] + sum(8 * n[j] for j in range(1, k))          # bounds read / written once (windows stay in shared memory)
            continue
        groups = 1 if k == net.L + 1 else -(-n[k] // 64)
        top = net.L if k == net.L + 1 else k
        for j in range(top, 0, -1):                   # A_j^T: layer j -> layer j - 1
            flop += groups * 2 * 64 * mac[j - 1]
            byts += groups * 256 * (n[j] + 3 * n[j - 1])
    peaks = load_peaks()
    return {'value': world * children / dt, 'unit': 'children/s', 'n_gpus': world, 'parents_per_step': parents, 'steps': steps, 'ms_per_step': dt / steps * 1e3,
            'launches_per_step': launches // steps, 'second_kw_passes': second, 'infeasible_children_dropped': infeasible, 'queue_domains_at_end': len(fs.queue),
            'api': 'FrontierStep.step: gnnb_queue_pick -> split -> gnnb_child_bounds -> gnnb_score -> gnnb_queue_add, all device-resident',
            'host_traffic': 'three counts read back per step (picked, second-pass domains, added); no bounds, masks or scores cross PCIe',
            'lp': 'surrogate (no Gurobi): lower bound = KW / interval bound of the property output, zero duals, primals = activations of the ball centre',
            'child_bounds': {'value': n2 / (cb_ms * 1e-3), 'unit': 'children/s', 'ms_per_call': cb_ms, 'children': n2,
                             'executed_gflop_per_child': flop / 1e9, 'achieved_tflops': flop * n2 / (cb_ms * 1e-3) / 1e12,
                             'roofline': {'bound': 'hbm', 'achieved': byts * n2 / (cb_ms * 1e-3) / 1e9, 'peak': peaks['gbs'], 'unit': 'GB/s',
                                          'frac': byts * n2 / (cb_ms * 1e-3) / 1e9 / peaks['gbs'], 'traffic': None,
                                          'note': 'bytes of the executed schedule (dense layers: [n, 64] column blocks as 256-byte-per-row tile images written '
                                                  'and re-read by every transposed-propagation and reduction launch), not compulsory bytes; the windowed '
                                                  'conv-layer kernel is issue-bound (ncu: 72 % of issue slots, no DRAM traffic to speak of, '
                                                  'profiles/r03t_ncu_kw_cone.txt)'},
                             'note': 'bounds part of KWConvGen.update_the_model (plnn/conv_kwinter_gen.py:558-660) for a batch of children: KW recursion '
                                     '(windowed fp32 kernel for conv layers; the linear layers and the property output as 64-column blocks through the '
                                     'tensor-core propagation kernel, fp16 x 3) + interval pass + masks'}}



def load_peaks():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except (OSError, ValueError):
        pass
    # a short timed region runs at burst clocks, a long one under the power cap (profiling recipe): bf16 burst / sustained
    return {'tf_sustained': peaks.get('bf16_tflops_sustained', 1400.0), 'tf_burst': peaks.get('bf16_tflops', 1650.0),
            'gbs': peaks.get('hbm_gbs', 6650.0),
            'source': 'MEASURED_PEAKS.json hbm_gbs / bf16_tflops (burst) / bf16_tflops_sustained (of measured)' if peaks else
                      'B200_PROFILING.md fallback 6.65 TB/s / 1.65 PF burst / 1.4 PF sustained (of fallback)'}


def roofline_of(net, fr, m, n_domains, world, scorer, peaks):
    """roofline object of one measured workload (dominant kernel class, live CUDA-event times, whole-path figures)."""
    timed_s = m['ms'] * 1e-3
    peak_tf = peaks['tf_burst'] if timed_s < 0.25 else peaks['tf_sustained']        # which bf16 peak applies to this timed region
    r = kernel_rooflines(net, fr, m['prof'], n_domains, T=2, peak_tf=peak_tf, peak_gbs=peaks['gbs'])
    r['peak_source'] = peaks['source'] + (' - tensor peak: burst (timed region %.0f ms)' % (timed_s * 1e3) if timed_s < 0.25
                                          else ' - tensor peak: sustained (timed region %.0f ms)' % (timed_s * 1e3))
    r['timing'] = ('CUDA events around every launch on the launching stream, over a second pass of the same steps '
                   '(the events serialise launches, so `value` is timed without them)')
    flops_dom = net.flops_per_domain()
    r['whole_path'] = {'flop_per_subdomain': flops_dom, 'achieved_tflops': m['value'] / world * flops_dom / 1e12,
                       'frac_of_bf16_peak': m['value'] / world * flops_dom / 1e12 / peak_tf, 'bf16_peak_used': peak_tf,
                       'hbm_bytes_per_subdomain': r.pop('_bytes_per_subdomain'),
                       'note': 'fp32 accuracy needs 3 fp16 MMA passes per product: the tensor ceiling is 1/3 of the bf16 peak'}
    try:      # DRAM bytes per launch of that kernel class from the committed ncu --set full capture, scaled to this run's wave size
        kt = json.load(open(os.path.join(ROOT, 'profiles', 'kernel_traffic.json')))
        wave = min(fr.B, scorer.get_option('chunk') or 1024)          # subdomains per launch (gnnb_api.cu: waves of `chunk`, default 1 024)
        r['traffic'] = kt[r['kernel_class']]['dram_bytes_per_launch_per_subdomain'] * wave
        r['traffic_source'] = kt['_source']
    except (OSError, ValueError, KeyError):
        r['traffic'] = None
    return r


def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from gnn_branching_b200 import GraphNet, synthetic_frontier
    from gnn_branching_b200.dist import gather_winner_records

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: the scoring path has no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    # N = 1: BASELINE configs[1..3] (base x 1 024, or --workload wide / deep x 4 096).  N > 1: BASELINE configs[4], the 65 536-
    # subdomain base frontier sharded contiguously over the N GPUs (strong scaling: the total is fixed)
    strong = world > 1 and not args.domains and args.workload == 'base'
    B = args.domains or (FRONTIER_TOTAL // world if strong else DEFAULT_DOMAINS[args.workload])
    K, W = args.steps, max(args.warmup, 0)

    net, lbs, ubs, wp, bp = load_problem(args.workload)
    sd = load_weights(args.weights)
    model = GraphNet(2, 64, math=args.math, chunk=args.chunk)
    model.load_state_dict(sd)
    model = model.eval().to(dev)
    if world > 1:      # the GNN parameters are broadcast once from rank 0 (SURVEY §8e), outside the timed region
        from gnn_branching_b200.dist import broadcast_gnn_weights
        broadcast_gnn_weights(model, src=0)
    # two different frontiers used alternately: with the workspace they exceed the 126 MB L2 several times over (a frontier of
    # more than 8 192 subdomains is > 1 GB of inputs on its own: one is enough)
    n_fronts = 2 if B <= 8192 else 1
    fronts = [synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=1000 * (7 + rank) + i, device=dev) for i in range(n_fronts)]
    scorer = model.scorer(local)
    for kv in args.opt:
        key, val = kv.split('=')
        scorer.set_option(key, int(val))
    math_mode = {0: 'tc', 1: 'simt'}[scorer.get_option('math')]

    m = measure_device(scorer, fronts, B, K, W, world, dev, local, gather_winner_records)
    value, ms, launches, clocks = m['value'], m['ms'], m['launches'], m['clocks']
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *m['outputs'])

    # ---- end to end through the public API with pinned HOST buffers (copies inside the timed region) ----
    e2e = None
    if not args.no_e2e:
        host_fronts = [f.cpu().pin() for f in fronts]
        e2e = measure_e2e(model, host_fronts, B, K, W, world, dev, gather_winner_records)
        del host_fronts

    # ---- the device-resident branch-and-bound step (every rank takes part: its own queue, its own subtree) ----
    fstep = None
    if not args.no_step and not args.domains and math_mode == 'tc':
        try:
            fstep = measure_frontier_step(model, args.workload, dev, world)
            scorer.set_network(net, key=net.key)
        except Exception as e:              # a secondary object must never take the headline down
            fstep = {'error': repr(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    peak_gbs = peaks['gbs']
    roofline = roofline_of(net, fronts[0], m, K * B, world, scorer, peaks)

    # ---- B = 1 latency (the reference's native usage: one subdomain per call, plnn/relu_conv_gnnkwthreshold.py:117) ----
    b1 = None
    if world == 1:
        one = fronts[0].slice(0, 1).contiguous()
        one_host = one.cpu().pin()
        for _ in range(5):
            scorer.score(one, return_scores=False, check=False)
            model.score_frontier(one_host, return_scores=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            scorer.score(one, return_scores=False, check=False)
        e1.record()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(50):
            model.score_frontier(one_host, return_scores=False)
        torch.cuda.synchronize()
        b1 = {'device_ms': e0.elapsed_time(e1) / 50, 'e2e_ms': (time.perf_counter() - t0) / 50 * 1e3,
              'note': 'one subdomain per call; device_ms: inputs resident, CUDA events; e2e_ms: pinned host inputs, winners read back'}
        del one, one_host

    # ---- BASELINE configs[2] and [3] (wide / deep x 4 096) as secondary objects of the default line ----
    others = {}
    if world == 1 and args.workload == 'base' and not args.domains and not args.no_secondary:
        del fronts
        torch.cuda.empty_cache()
        for wl in ('wide', 'deep'):
            try:
                net2, lbs2, ubs2, wp2, bp2 = load_problem(wl)
                B2 = DEFAULT_DOMAINS[wl]
                fr2 = [synthetic_frontier(net2, lbs2, ubs2, wp2, bp2, B2, seed=1000 * (17 + i) + len(wl), device=dev) for i in range(2)]
                m2 = measure_device(scorer, fr2, B2, 20, 3, 1, dev, local, gather_winner_records)
                hf2 = [fr2[0].cpu().pin()]
                e2 = measure_e2e(model, hf2, B2, 3, 1, 1, dev, gather_winner_records)
                del hf2
                others[wl] = {'value': m2['value'], 'unit': UNIT, 'ms_per_step': m2['ms'] / 20, 'steps': 20, 'warmup': 3,
                              'workload': f'cifar_{wl}_kw x {B2} synthetic subdomains per step', 'gpu_launches': m2['launches'],
                              'clocks': m2['clocks'], 'e2e': e2, 'roofline': roofline_of(net2, fr2[0], m2, 20 * B2, 1, scorer, peaks)}
                del fr2
                torch.cuda.empty_cache()
            except Exception as e:          # a secondary object must never take the headline down
                others[wl] = {'error': repr(e)[:300]}
        fronts = [synthetic_frontier(net, lbs, ubs, wp, bp, B, seed=1000 * (7 + rank) + i, device=dev) for i in range(n_fronts)]
        scorer.set_network(net, key=net.key)

    # ---- the BaBSR / KW heuristic on the same frontier (SURVEY §8f rank 1; secondary line, not the headline metric) ----
    babsr = None
    if world == 1 and not args.no_babsr:
        from gnn_branching_b200 import babsr_frontier
        fr0 = fronts[0]
        for _ in range(3):
            babsr_frontier(fr0, scorer=scorer)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(20):
            babsr_frontier(fronts[i % 2], scorer=scorer)
        e1.record()
        torch.cuda.synchronize()
        bms = e0.elapsed_time(e1) / 20
        bbytes = B * (sum(net.hidden_sizes) * 12 + net.hidden_sizes[-1] * 4 + 16)      # l, u, mask per ReLU; Wp; outputs
        babsr = {'value': B / (bms * 1e-3), 'unit': UNIT, 'ms_per_call': bms, 'subdomains': B,
                 'roofline': {'bound': 'hbm', 'achieved': bbytes / (bms * 1e-3) / 1e9, 'peak': peak_gbs, 'unit': 'GB/s',
                              'frac': bbytes / (bms * 1e-3) / 1e9 / peak_gbs},
                 'note': 'choose_node_conv (plnn/kw_score_conv.py:41-156) batched, one thread block per subdomain, device-resident inputs'}
        if not args.no_cpu_baseline:
            from oracle import babsr_oracle as BO
            fc = fr0.slice(0, 64).cpu().contiguous()
            order = [0] + list(range(1, net.L))
            t0 = time.perf_counter()
            for _ in range(3):
                sc_, ic_ = BO.babsr_scores(fc)
                BO.babsr_decide(sc_, ic_, fc.mask, net.hidden_sizes, [0] * 64, order, 0)
            babsr['cpu_baseline'] = {'value': 3 * 64 / (time.perf_counter() - t0), 'unit': UNIT, 'kind': 'port', 'cores': os.cpu_count(),
                                     'sample': '64 subdomains x 3 passes, oracle/babsr_oracle.py (batched scores, per-domain decision rule)'}

    # ---- one online fine-tuning step (SURVEY §8f rank 2; secondary line): gradient of gnn_score - kw_score + Adam, B = 1 ----
    online = None
    if world == 1 and not args.no_online:
        one = fronts[0].slice(0, 1)
        cand = one.mask[0].nonzero().view(-1).tolist()
        if len(cand) >= 2:
            terms = [(0, cand[0], 1.0), (0, cand[-1], -1.0)]
            saved = scorer.weights()
            for _ in range(2):
                scorer.score_grad(one, terms)
                scorer.adam_step(1e-4, weight_decay=1e-4)
            torch.cuda.synchronize()
            l0, t0 = scorer.launches, time.perf_counter()
            for _ in range(10):
                scorer.score_grad(one, terms)
                scorer.adam_step(1e-4, weight_decay=1e-4)
            torch.cuda.synchronize()
            oms = (time.perf_counter() - t0) / 10 * 1e3
            online = {'ms_per_step': oms, 'steps_per_s': 1e3 / oms, 'launches_per_step': (scorer.launches - l0) // 10,
                      'note': 'GraphChoice.online_learning (graph_score_online.py:62-77): fp32 forward with tape + backward + Adam + '
                              'repack of the tensor-core weight planes, one subdomain, wall clock around the C-ABI calls'}
            scorer.adam_reset()
            scorer.set_gnn(saved, key=None)       # the headline numbers above were measured before; restore anyway
            if not args.no_cpu_baseline:
                from oracle.online_oracle import OnlineOracle
                oo = OnlineOracle(load_weights(args.weights))
                oc = one.cpu().contiguous()
                oo.online_learning(oc, cand[0], [0, 0], 1.0)
                t0 = time.perf_counter()
                for _ in range(3):
                    oo.online_learning(oc, cand[0], [0, 0], 1.0)
                online['cpu_baseline'] = {'ms_per_step': (time.perf_counter() - t0) / 3 * 1e3, 'kind': 'port', 'cores': os.cpu_count(),
                                          'sample': '3 steps, oracle/online_oracle.py (torch autograd + torch.optim.Adam on the host cores)'}

    # ---- the device-resident domain queue (SURVEY §8f rank 4; secondary line): add / pick of whole frontiers ----
    queue = None
    if world == 1 and not args.no_queue:
        from gnn_branching_b200 import DomainQueue, DomainBatch
        f0 = fronts[0]
        Bq = min(B, 1024)
        g = torch.Generator(device='cpu').manual_seed(3)
        batch = DomainBatch((torch.randn(Bq, generator=g) - 1.0).to(dev), torch.zeros(Bq, device=dev), [t[:Bq] for t in f0.lb],
                            [t[:Bq] for t in f0.ub], (f0.mask[:Bq] * -1).to(torch.int8), torch.zeros(Bq, 2, dtype=torch.int32, device=dev))
        q = DomainQueue(scorer, capacity=4 * Bq)
        for _ in range(2):
            q.add(batch); q.pick(Bq, float('inf'))
        torch.cuda.synchronize()
        reps, t_add, t_pick = 10, 0.0, 0.0
        for _ in range(reps):
            t0 = time.perf_counter(); q.add(batch); torch.cuda.synchronize(); t_add += time.perf_counter() - t0
            t0 = time.perf_counter(); out = q.pick(Bq, float('inf')); torch.cuda.synchronize(); t_pick += time.perf_counter() - t0
        row_bytes = 2 * 4 * (net.n0 + net.n_hidden + 1) + net.n_hidden + 16
        queue = {'domains': Bq, 'add_domains_per_s': Bq * reps / t_add, 'pick_domains_per_s': Bq * reps / t_pick,
                 'payload_bytes_per_domain': row_bytes,
                 'add_gbs': 2 * row_bytes * Bq * reps / t_add / 1e9, 'pick_gbs': 2 * row_bytes * Bq * reps / t_pick / 1e9, 'peak_gbs': peak_gbs,
                 'note': 'add_domain / pick_out of plnn/branch_and_bound.py:159-184 for a whole frontier per call: payload rows copied '
                         'once into / out of the device pool (read + write counted), order kept by a radix sort of (key, slot) pairs; '
                         'wall clock around the C-ABI calls, which read one count back per call'}
        del q, out

    cb = None
    if not args.no_cpu_baseline and world == 1:
        cb, _ = cpu_baseline(args.workload, args.weights)
        # the reference's native deployment is eager PyTorch on the GPU (graph_score.py:13): the unmodified module (oracle/_ref)
        # with CUDA tensors at B = 1 (its native usage), 32 and 1 024 — library kernels, a reported baseline like the CPU figure
        eg = _run_ref_runner('cuda', args.workload, args.weights, (1, 32, 1024), 3, 1, timeout=600)
        if eg and 'error' not in eg:
            cb['eager_pytorch_on_gpu'] = {'value': eg['value'], 'unit': UNIT, 'best_batch': eg['best_batch'], 'b1_latency_ms': eg['b1_latency_ms'],
                                          'rate_by_batch': {k: v['rate'] for k, v in eg['per_batch'].items()}, 'kind': 'reference',
                                          'note': 'unmodified graphnet/graph_conv.py GraphNet.forward (oracle/_ref) on this B200, torch eager '
                                                  '(cuDNN / cuBLAS kernels), own process'}
        else:
            cb['eager_pytorch_on_gpu'] = eg or {'error': 'oracle/_ref is not staged'}

    wl_name = (f'cifar_base_kw frontier of {B * world} synthetic subdomains sharded across {world} GPUs ({B} per GPU per step)' if strong
               else f'cifar_{args.workload}_kw x {B} synthetic subdomains per GPU per step')
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'strong' if strong else 'weak', 'vs_baseline': None,
            'dtype': 'fp16x3 (fp32 accumulate)' if math_mode == 'tc' else 'f32', 'data': 'synthetic',
            'config': {'workload': wl_name, 'gnn': 'GraphNet(T=2,p=64)', 'weights': args.weights, 'math': math_mode,
                       'chunk': min(B, scorer.get_option('chunk') or 1024), 'fuse': scorer.get_option('fuse'),
                       'l2': f'{n_fronts} frontier(s) of {B} subdomains used alternately; inputs + per-wave workspace exceed the 126 MB L2',
                       'sharding': f'{world} ranks x {B} subdomains, winners all-gathered (8 B/subdomain)'},
            'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches, 'roofline': roofline, 'cpu_baseline': cb,
            'b1_latency_ms': b1, 'wide': others.get('wide'), 'deep': others.get('deep'),
            'babsr': babsr, 'online': online, 'queue': queue, 'frontier_step': fstep}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
