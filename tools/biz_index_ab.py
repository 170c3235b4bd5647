"""Developer tool: the business index against the grouped business path, in one process.

Two handles on the same graph (default: C2 at full size): one with the business index, one created
with BLP_BIZ_INDEX=0 (the grouped path: counting sort, per-group hop-2 expansion, un-permute).
Calls alternate between the two, each preceded by a 256 MiB write that flushes the L2 (as bench.py
does), and are timed with CUDA events: the business side alone (score_side) and the whole step
(score_pairs, both sides on one stream).  Every output column of the two handles is compared with
torch.equal.  Prints one JSON line with the card's name and power limit, read in the same run.
usage: biz_index_ab.py [--config C2] [--reps 10] [--out FILE]
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                            '--format=csv,noheader', '-i', '0'], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        return 'unknown (%r)' % exc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='C2')
    ap.add_argument('--pairs', type=int, default=None)
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch
    lib = importlib.import_module('bipartite-link-prediction_b200._lib')
    graph = importlib.import_module('bipartite-link-prediction_b200.graph')
    synth = importlib.import_module('bipartite-link-prediction_b200.synth')
    cfg, eu, eb, pu, pv = synth.make_config(a.config, n_pairs=a.pairs)
    handles = {}
    build_s = {}
    for name, env in (('index', None), ('grouped', '0')):
        os.environ.pop('BLP_BIZ_INDEX', None)
        if env is not None:
            os.environ['BLP_BIZ_INDEX'] = env
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        handles[name] = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, device=0)
        build_s[name] = time.perf_counter() - t0
    os.environ.pop('BLP_BIZ_INDEX', None)
    du, dv = torch.from_numpy(pu).cuda(), torch.from_numpy(pv).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    outs = {k: None for k in handles}

    def timed(fn):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1), r

    biz = {k: [] for k in handles}
    biz_stats = {k: [] for k in handles}
    step = {k: [] for k in handles}
    for it in range(a.reps + 2):                     # the first two rounds are warm-up
        for name, G in handles.items():
            ms, _ = timed(lambda: G.score_side(lib.SIDE_BUSINESS, du, dv))
            st = G.score_stats(lib.SIDE_BUSINESS)
            ms_step, outs[name] = timed(lambda: G.score_pairs(du, dv, out=outs[name], concurrent=False))
            if it >= 2:
                biz[name].append(ms)
                biz_stats[name].append(st['group_ms'] + st['score_ms'])
                step[name].append(ms_step)
    torch.cuda.synchronize()
    equal = {k: bool(torch.equal(outs['index'][k], outs['grouped'][k])) for k in outs['index']}
    res = {'config': a.config, 'pairs': int(pu.size), 'reps': a.reps, 'card': card(),
           'columns_equal': equal, 'all_equal': all(equal.values()),
           'index_info': {k: handles['index'].info()[k] for k in ('biz_index_bytes', 'biz_index_build_ms')},
           'graph_create_s': build_s}
    for name in handles:
        res[name] = {'business_side_ms_median': statistics.median(biz[name]),
                     'business_side_ms': biz[name],
                     'business_stats_group_plus_score_ms_median': statistics.median(biz_stats[name]),
                     'step_ms_median': statistics.median(step[name]), 'step_ms': step[name],
                     'path': handles[name].score_stats(lib.SIDE_BUSINESS)['path']}
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
