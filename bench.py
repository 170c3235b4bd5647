#!/usr/bin/env python
"""bench.py -- candidate pairs scored per second on Yelp-shaped synthetic inputs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C2|C3|C4|C5] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: every pair of the workload gets the seven
reference outputs (u_cn,u_jaccard,u_adamic,b_cn,b_jaccard,b_adamic,pa; the two union sizes are
computed as well where a buffer is given).

N=1 workload: BASELINE.json configs[1] ("C2": 366k users x 61k businesses, 1.5M reviews, 10M
candidate pairs).  --config C3 / C4 / C5 select the other BASELINE.json configs (C5: one GPU's
eighth of the 1B pairs).

N>1: weak scaling through the product's multi-GPU API.  ONE pair list of N x 10M pairs (the
concatenation of N shards, each drawn exactly like the N=1 workload) is cut with
dist.shard_bounds into user-aligned, work-balanced slices; the adjacency is replicated; every rank
scores its slice with the columns of rank 0's peer-mapped dist.ResultWindow as the kernels' output
arrays, so the result rows cross NVLink from inside the scoring kernels and the timed region ends
with every row of the whole list resident on rank 0 (`value`).  Beside it: the same scoring into
local memory (`scoring_only`) and local scoring followed by a grouped NCCL send/recv gather
(`nccl_gather`, the baseline the fused path is measured against).  Afterwards rank 0 compares ALL
rows with its own unsharded call and a sample with the C oracle.

One JSON line on stdout (rank 0).  `value` is device-resident throughput (CUDA events, max over
ranks); `e2e` goes through the host-buffer API (pinned H2D of the pair ids, D2H of the seven
reference outputs, 48 B/pair); `roofline` is the user-side scoring kernel (the dominant one)
against MEASURED_PEAKS.json; `cpu_baseline` is the reference's algorithm on the host: the headline
figure is ONE process (the reference is single-threaded) of the line-for-line restatement with set
membership ("fair", BASELINE.md section 2) on a C2 subsample; the faithful list-membership form,
the reference's own code (oracle/_ref) on C1, the vectorised oracle and the plain-C port (one
thread / every core, the latter over ALL pairs and compared with the GPU's output) sit beside it.
`--impl reference` prints the all-core CPU arm as its own line.

`--dump-outputs DIR` writes what the last timed step computed -- every column the timed call
returns (N>1: rank 0's window) -- as DIR/<column>.npy in float64, which holds the integer columns
exactly.  Above DUMP_ROWS rows it writes a fixed seeded sample of rows, the same for every run with
the same arguments; DIR/row_index.npy says which.  Two builds can so be compared output for output.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree, which may be read-only
PKG = 'bipartite-link-prediction_b200'
METRIC = 'candidate pairs scored/sec'
UNIT = 'pairs/s'
METHODS = ['common_neighbors', 'jaccard', 'adamic_adar']
NOTE = ('reference _snap.so (Python 2) unavailable -- the CPU baseline is a line-for-line '
        "re-execution of similarity.py's formulas (oracle/similarity_oracle.py); the reference's own "
        'similarity.py (oracle/_ref: bytecode of the unmodified functions + a SNAP stand-in) is timed '
        'on C1 beside it and agrees with it row for row')


def pkg(sub):
    return importlib.import_module(PKG + '.' + sub)


# ------------------------------------------------------------------------------------ CPU arm
_G = None
_EX = None


def _cpu_worker(args):
    side, keys = args
    from oracle import similarity_oracle as oa
    ex = {k: _EX[k] for k in keys}
    t = time.perf_counter()
    if side == 'u':
        oa.users(ex, _G, METHODS, [None] * 3, write=False)
    else:
        oa.business(ex, _G, METHODS, [None] * 3, write=False)
    return time.perf_counter() - t


def _cpu_worker_packed(args):
    side, ex = args
    from oracle import similarity_oracle as oa
    t = time.perf_counter()
    oa.business(ex, _G, METHODS, [None] * 3, write=False)
    return time.perf_counter() - t


def _samples(pu, pv, n_user_groups, n_biz_groups):
    """Structure-preserving samples: ALL pairs of the first n example users (hop2(u) amortised over
    the same K pairs as in the full run) / ALL pairs of n seeded-random candidate businesses."""
    ok = (pu >= 0) & (pv >= 0)
    users_sorted = np.unique(pu[ok])
    sel_u = ok & np.isin(pu, users_sorted[:n_user_groups])
    rng = np.random.default_rng(7)
    bizs = np.unique(pv[ok])
    sel_b = ok & np.isin(pv, rng.choice(bizs, size=min(n_biz_groups, bizs.size), replace=False))
    return sel_u, sel_b


def cpu_reference_all_cores(cfg, eu, eb, pu, pv, n_user_groups, n_biz_groups, procs):
    """Oracle A (set membership) on every host core over structure-preserving samples; the two
    per-pair costs add: rate = 1 / (t_u/S_u + t_b/S_b).  Graph loading is not timed."""
    global _G, _EX
    import multiprocessing as mp
    from oracle import similarity_oracle as oa
    synth = pkg('synth')
    n_users = cfg['n_users']
    ids_eu, ids_eb = synth.shared_ids(n_users, eu, eb)
    _G = oa.MiniSnapGraph.from_edges(zip(ids_eu.tolist(), ids_eb.tolist()))
    ctx = mp.get_context('fork')

    def run(side, sel):
        global _EX
        ids_pu, ids_pv = synth.shared_ids(n_users, pu[sel], pv[sel])
        _EX = synth.examples_dict(ids_pu, ids_pv)
        keys = list(_EX.keys())
        if side == 'b':
            # shard by business so that every hop2(v) is built once, as in one process
            byb = {}
            for u in keys:
                for v in _EX[u]:
                    byb.setdefault(v, []).append(u)
            bl = list(byb.keys())
            full = _EX
            packs = []
            for p in range(procs):
                mine = set(bl[p::procs])
                us = set()
                for v in mine:
                    us.update(byb[v])
                packs.append({u: {v: 0 for v in full[u] if v in mine} for u in sorted(us)})
            t0 = time.perf_counter()
            with ctx.Pool(procs) as pool:
                pool.map(_cpu_worker_packed, [('b', pk) for pk in packs])
            return time.perf_counter() - t0, int(sel.sum())
        shards = [keys[p::procs] for p in range(procs)]
        t0 = time.perf_counter()
        with ctx.Pool(procs) as pool:
            pool.map(_cpu_worker, [(side, sh) for sh in shards])
        return time.perf_counter() - t0, int(sel.sum())

    sel_u, sel_b = _samples(pu, pv, n_user_groups, n_biz_groups)
    t_u, s_u = run('u', sel_u)
    t_b, s_b = run('b', sel_b)
    rate = 1.0 / (t_u / s_u + t_b / s_b)
    sample = ('user side: all %d pairs of the first %d example users in %.1fs; business side: all '
              '%d pairs of %d seeded-random candidate businesses in %.1fs; combined as '
              '1/(t_u/S_u+t_b/S_b); %d processes; graph load untimed' %
              (s_u, n_user_groups, t_u, s_b, n_biz_groups, t_b, procs))
    _G = None
    _EX = None
    return rate, sample, {'user_pairs_per_s': s_u / t_u, 'business_pairs_per_s': s_b / t_b}


def cpu_single_process(cfg, eu, eb, pu, pv, n_user_groups, n_biz_groups):
    """BASELINE.md section 2, the figure the >=100x target is judged against: ONE process of the
    line-for-line restatement with set membership ("fair") on a subsample of this workload."""
    from oracle import similarity_oracle as oa
    synth = pkg('synth')
    n_users = cfg['n_users']
    ids_eu, ids_eb = synth.shared_ids(n_users, eu, eb)
    G = oa.MiniSnapGraph.from_edges(zip(ids_eu.tolist(), ids_eb.tolist()))
    sel_u, sel_b = _samples(pu, pv, n_user_groups, n_biz_groups)
    out = []
    for side, sel in (('u', sel_u), ('b', sel_b)):
        ids_pu, ids_pv = synth.shared_ids(n_users, pu[sel], pv[sel])
        ex = synth.examples_dict(ids_pu, ids_pv)
        t0 = time.perf_counter()
        (oa.users if side == 'u' else oa.business)(ex, G, METHODS, [None] * 3, write=False)
        out.append((time.perf_counter() - t0, int(sel.sum())))
    (t_u, s_u), (t_b, s_b) = out
    rate = 1.0 / (t_u / s_u + t_b / s_b)
    sample = ('ONE process, set membership; user side: all %d pairs of the first %d example users in '
              '%.1fs; business side: all %d pairs of %d seeded-random candidate businesses in %.1fs; '
              'combined as 1/(t_u/S_u+t_b/S_b); graph load untimed' %
              (s_u, n_user_groups, t_u, s_b, n_biz_groups, t_b))
    return rate, sample, {'user_pairs_per_s': s_u / t_u, 'business_pairs_per_s': s_b / t_b}


def cpu_c1_legs(n_example_users=300):
    """BASELINE.json configs[0] (the reference's own CPU-runnable case), one process: the faithful
    form (node ids in a LIST, similarity.py:22,52), the fair form, the reference's OWN code
    (oracle/_ref) and the vectorised oracle."""
    from oracle import algebra_oracle as ob
    from oracle import ref_runner as rr
    from oracle import similarity_oracle as oa
    synth = pkg('synth')
    cfg, eu, eb, pu, pv = synth.make_config('C1')
    ids_eu, ids_eb = synth.shared_ids(cfg['n_users'], eu, eb)
    G = oa.MiniSnapGraph.from_edges(zip(ids_eu.tolist(), ids_eb.tolist()))
    ok = (pu >= 0) & (pv >= 0)
    sel = ok & np.isin(pu, np.unique(pu[ok])[:n_example_users])
    ids_pu, ids_pv = synth.shared_ids(cfg['n_users'], pu[sel], pv[sel])
    ex = synth.examples_dict(ids_pu, ids_pv)
    s = int(sel.sum())
    legs = {'c1_sample': 'all %d pairs of the first %d example users of C1 (10k x 2k, 50k review '
                         'lines), both sides, three methods each, one process' % (s, n_example_users)}
    res = {}
    for name, faithful in (('fair', False), ('faithful', True)):
        t0 = time.perf_counter()
        ru = oa.users(ex, G, METHODS, [None] * 3, write=False, faithful=faithful)
        rb = oa.business(ex, G, METHODS, [None] * 3, write=False, faithful=faithful,
                         reproduce_reference_bug=True)
        legs['c1_%s_pairs_per_s' % name] = s / (time.perf_counter() - t0)
        res[name] = (ru, rb)
    if rr.available():
        with tempfile.TemporaryDirectory() as d:
            t0 = time.perf_counter()
            rr.users_business(ex, G, d)
            legs['c1_reference_own_code_pairs_per_s'] = s / (time.perf_counter() - t0)
            files = [json.load(open(os.path.join(d, n + '.json')))
                     for n in ('u_cn', 'u_jaccard', 'u_adamic', 'b_cn', 'b_jaccard', 'b_adamic')]
        ru, rb = res['faithful']
        same = True
        for got, want in zip(files, list(ru) + list(rb)):
            for u in want:
                for v in want[u]:
                    x, y = got[u][v], want[u][v]
                    same = same and (x == y or abs(x - y) <= 1e-12 * abs(y)) and type(x) is type(y)
            same = same and got.keys() == dict(want).keys()
        legs['c1_reference_own_code_equals_restatement'] = bool(same)
        legs['c1_reference_own_code'] = ('oracle/_ref: the reference\'s similarity.py users()+business() '
                                         'executed as they are (list membership, per-pair prints '
                                         'swallowed, JSON dumps included), SNAP stand-in')
    else:
        legs['c1_reference_own_code'] = 'oracle/_ref not built on this machine'
    t0 = time.perf_counter()
    ob.score_pair_arrays(cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv)
    legs['c1_vectorised_oracle_b_pairs_per_s'] = pu.size / (time.perf_counter() - t0)
    legs['c1_vectorised_sample'] = 'all %d pairs of C1, scipy.sparse algebra, one process' % pu.size
    return legs


def cpu_c_port(cfg, eu, eb, pu, pv, cores):
    """The plain-C restatement: one thread on the first 1M pairs, then ALL pairs on every core
    (its output is kept and compared with the GPU's)."""
    from oracle import c_oracle
    sides = {}
    m = min(int(pu.size), 1_000_000)
    t0 = time.perf_counter()
    c_oracle.score_pair_arrays(cfg['n_users'], cfg['n_biz'], eu, eb, pu[:m], pv[:m])
    sides['c_port_1thread_pairs_per_s'] = m / (time.perf_counter() - t0)
    sides['c_port_sample'] = 'first %d pairs, graph build included' % m
    t0 = time.perf_counter()
    full = c_oracle.score_pair_arrays_parallel(cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv,
                                               threads=cores)
    sides['c_port_all_cores_pairs_per_s'] = int(pu.size) / (time.perf_counter() - t0)
    sides['c_port_all_cores_sample'] = ('all %d pairs in %d contiguous slices, one thread each, '
                                        'graph build included in every slice' % (pu.size, cores))
    return sides, full


def compare_with_oracle(host, want):
    """Bit-exact integers and jaccard, adamic within 1e-8 relative (bar: 1e-6)."""
    bad = {}
    for k in ('u_cn', 'b_cn', 'pa', 'u_union', 'b_union'):
        if k in host:
            d = int((host[k].astype(np.int64) != want[k].astype(np.int64)).sum())
            if d:
                bad[k] = d
    for k in ('u_jaccard', 'b_jaccard'):
        if k in host:
            d = int((host[k] != want[k]).sum())
            if d:
                bad[k] = d
    worst = 0.0
    for k in ('u_adamic', 'b_adamic'):
        if k in host:
            nz = want[k] != 0
            if ((host[k] == 0) != (want[k] == 0)).any():
                bad[k] = 'zero pattern'
            if nz.any():
                worst = max(worst, float(np.max(np.abs(host[k][nz] - want[k][nz]) / want[k][nz])))
    if worst > 1e-8:
        bad['adamic_rel'] = worst
    return {'rows': int(len(want['pa'])), 'mismatches': bad, 'adamic_max_rel_err': worst,
            'ok': not bad}


# --dump-outputs: at most 2^19 rows of each of at most ten arrays, 8 B each: 42 MB in all
DUMP_ROWS = 1 << 19


def dump_rows(n):
    """The rows --dump-outputs writes: all n, or a fixed seeded sample of DUMP_ROWS, ascending."""
    if n <= DUMP_ROWS:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(n, size=DUMP_ROWS, replace=False))


def dump_outputs(path, cols, rows):
    """cols: column name -> device tensor of every row; writes rows `rows` of each as float64."""
    import torch
    os.makedirs(path, exist_ok=True)
    t_rows = torch.from_numpy(rows).to(next(iter(cols.values())).device)
    np.save(os.path.join(path, 'row_index.npy'), rows.astype(np.float64))
    for k, v in cols.items():
        np.save(os.path.join(path, k + '.npy'), v[t_rows].cpu().numpy().astype(np.float64))


# ------------------------------------------------------------------------------------ clocks
class ClockSampler(object):
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '50'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def wait_first(self, timeout=5.0):
        """nvidia-smi needs a moment before its first line: do not start timing without one."""
        t_end = time.perf_counter() + timeout
        while self.proc is not None and not self.rows and time.perf_counter() < t_end:
            time.sleep(0.05)

    def window(self, t0, t1):
        # samples taken inside the timed region; a region shorter than the sampling interval
        # takes the samples that bracket it
        if self.proc is not None:
            time.sleep(0.12)
        rows = [r for t, r in self.rows if t0 <= t <= t1]
        if not rows:
            rows = [r for t, r in self.rows if t0 - 0.15 <= t <= t1 + 0.15] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in rows:
            f = [x.strip() for x in r.split(',')]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, f[4:8]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None,
                'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons),
                'samples': len(sm)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


def _profile_json(name):
    try:
        return json.load(open(os.path.join(ROOT, 'profiles', name)))
    except (OSError, ValueError):
        return None



# ------------------------------------------------------------------------------------ other configs
def other_config_line(name, n_pairs, steps, rank, world, dev, cores, peak):
    """A short line for another BASELINE.json config, beside the headline one.

    N=1: `n_pairs` pairs of the config on this GPU (a stated part of the config's list when the whole
    list would take minutes to generate).  N>1: the config's list cut N ways (strong scaling): every
    rank generates and scores ITS contiguous share of the example users (user-aligned by
    construction), all rows land in rank 0's peer window.  Timed like the headline (3 warm-ups,
    L2 flushed before every step, CUDA events, max over ranks); a strided sample of the rows as
    they sit on rank 0 is compared with the C oracle."""
    import torch
    import torch.distributed as dist
    graph, roofline, _lib, dmod, synth = pkg('graph'), pkg('roofline'), pkg('_lib'), pkg('dist'), pkg('synth')
    t_gen = time.perf_counter()
    cfg = dict(synth.CONFIGS[name])
    cfg['n_pairs'] = int(n_pairs)
    eu, eb = synth.make_graph(seed=0, **cfg)
    deg = synth.degrees(cfg['n_users'], cfg['n_biz'], eu, eb)
    pu, pv = synth.make_pairs(edge_u=eu, edge_b=eb, seed=1, deg=deg, rank=rank, world=world, **cfg)
    t_gen = time.perf_counter() - t_gen
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, device=dev.index)
    d_u, d_b = torch.from_numpy(pu).to(dev), torch.from_numpy(pv).to(dev)
    n = int(pu.size)
    counts = [n]
    if world > 1:
        t = torch.zeros(world, dtype=torch.int64, device=dev)
        t[rank] = n
        dist.all_reduce(t)
        counts = [int(x) for x in t.tolist()]
    n_total, lo = sum(counts), sum(counts[:rank])
    window = dmod.ResultWindow(G, n_total, columns=dmod.ALL_COLUMNS, dst=0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the whole pair list on rank 0 (it derives jaccard / pa for the peers' rows, and checks them)
    all_u = all_b = None
    if world > 1:
        longest = max(counts)
        pad_u = torch.full((longest,), -1, dtype=torch.int32, device=dev)
        pad_b = torch.full((longest,), -1, dtype=torch.int32, device=dev)
        pad_u[:n], pad_b[:n] = d_u, d_b
        g_u = torch.empty(world * longest, dtype=torch.int32, device=dev)
        g_b = torch.empty(world * longest, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(g_u, pad_u)
        dist.all_gather_into_tensor(g_b, pad_b)
        if rank == 0:
            keep = torch.cat([torch.arange(c, device=dev) + r * longest for r, c in enumerate(counts)])
            all_u, all_b = g_u[keep].contiguous(), g_b[keep].contiguous()
            window.attach_pairs(all_u, all_b, (lo, lo + n))
        del g_u, g_b, pad_u, pad_b

    tot, ku, kb = 0.0, [], []
    for it in range(3 + steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dmod.score_into_window(G, d_u, d_b, window, lo)
        if world > 1:
            dmod.rows_landed(G)
            if rank == 0:
                window.derive()
        e1.record()
        e1.synchronize()
        if it >= 3:
            tot += e0.elapsed_time(e1)
            ku.append(G.score_stats(_lib.SIDE_USER))
            kb.append(G.score_stats(_lib.SIDE_BUSINESS))
        elif it == 2:
            sync_all()
    sync_all()
    t = torch.tensor([tot], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    line = None
    if rank == 0:
        cols = window.tensors()
        if world > 1:
            pu_all, pv_all = all_u.cpu().numpy(), all_b.cpu().numpy()
        else:
            pu_all, pv_all = pu, pv
        idx = np.arange(0, n_total, max(1, n_total // 40_000))
        try:
            from oracle import c_oracle
            want = c_oracle.score_pair_arrays_parallel(cfg['n_users'], cfg['n_biz'], eu, eb, pu_all[idx],
                                                       pv_all[idx], threads=min(cores, 8))
            tidx = torch.from_numpy(idx).to(dev)
            chk = compare_with_oracle({k: cols[k][tidx].cpu().numpy() for k in cols}, want)
            chk['what'] = 'strided sample of the %d rows on rank 0 vs the C oracle' % n_total
        except Exception as exc:
            chk = {'error': repr(exc)}
        u_cn = cols['u_cn'][lo:lo + n].cpu().numpy()
        b_cn = cols['b_cn'][lo:lo + n].cpu().numpy()
        ab = roofline.algorithmic_bytes(cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv, u_cn, b_cn)
        ku_ms = statistics.mean(s['score_ms'] for s in ku)
        kb_ms = statistics.mean(s['score_ms'] for s in kb)
        bytes_u = ab['user'] + ab['pa']
        line = {'config': name, 'pairs_total': n_total, 'pairs_rank0': n, 'n_gpus': world,
                'scaling': 'strong' if world > 1 else None,
                'of_config': '%d of the config\'s %d pairs' % (n_total, synth.CONFIGS[name]['n_pairs']),
                'value': n_total / (ms * 1e-3), 'unit': UNIT, 'ms_per_step': ms, 'steps': steps,
                'user_side_ms': ku_ms, 'business_side_ms': kb_ms,
                'launch': {'ctas': ku[-1]['ctas'], 'threads_per_cta': ku[-1]['threads_per_cta'],
                           'smem_bytes': ku[-1]['smem_bytes'], 'range_passes': ku[-1]['range_passes']},
                'roofline': {'bound': 'hbm', 'kernel': 'user side (rank 0\'s share)', 'achieved': bytes_u / (ku_ms * 1e-3) / 1e9,
                             'peak': peak, 'unit': 'GB/s', 'frac': bytes_u / (ku_ms * 1e-3) / 1e9 / peak,
                             'algorithmic_bytes_per_launch': bytes_u,
                             'whole_step_achieved': ab['total'] / (ms * 1e-3) / 1e9},
                'parity_sample': chk, 'graph': G.info(), 'host_generation_s': t_gen}
    sync_all()
    window.close()
    G.close()
    return line

# ------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--config', default='C2')
    ap.add_argument('--pairs', type=int, default=None, help='pairs per GPU (default: config)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cpu-user-groups', type=int, default=None)
    ap.add_argument('--cpu-biz-groups', type=int, default=None)
    ap.add_argument('--no-other-configs', action='store_true',
                    help='skip the short C3 / C4 lines that follow the headline measurement')
    ap.add_argument('--derive', default=None, help="N>1: comma list of columns rank 0 derives (default pa)")
    ap.add_argument('--quick', action='store_true',
                    help='headline measurement and checks only: no comparison arms, no e2e, no other configs')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step to DIR/<column>.npy (float64; a '
                         'fixed seeded sample of %d rows when there are more)' % DUMP_ROWS)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl != 'b200':
        ap.error('--dump-outputs writes what the GPU path computed; it does not apply to --impl %s' % a.impl)

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if world == 1 and a.gpus > 1 and 'RANK' not in os.environ:
        # convenience: re-launch ourselves under torchrun
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1',
               '--nproc-per-node', str(a.gpus), '--master-addr', '127.0.0.1', '--master-port',
               os.environ.get('MASTER_PORT', '29511')] + sys.argv
        sys.exit(subprocess.call(cmd))
    if a.warmup < 3 and a.impl == 'b200':
        a.warmup = 3

    synth = pkg('synth')
    cfg = dict(synth.CONFIGS[a.config])
    # C5 is defined over 8 GPUs (1B pairs): one GPU's share is an eighth of the list
    per_gpu = a.pairs or (cfg['n_pairs'] // 8 if a.config == 'C5' else cfg['n_pairs'])
    workload = ('%s: %d users x %d businesses, %d review lines, %d candidate pairs per GPU '
                '(K=%d per example user), seeded synthetic Yelp-shaped' %
                (a.config, cfg['n_users'], cfg['n_biz'], cfg['n_reviews'], per_gpu, cfg['k']))
    config = {'workload': workload, 'name': a.config, 'pairs_per_gpu': per_gpu,
              'outputs_per_pair': 7, 'l2': 'L2 flushed (256 MiB write) before every timed step'}
    if world > 1:
        config['sharding'] = ('ONE list of %d x %d pairs (N shards drawn like the N=1 workload, '
                              'seed 1+shard, concatenated) cut by dist.shard_bounds into '
                              'user-aligned work-balanced slices; adjacency replicated; results of '
                              'every rank stored by the scoring kernels into rank 0\'s peer-mapped '
                              'window (NVLink) inside the timed region' % (world, per_gpu))
    cores = len(os.sched_getaffinity(0))

    eu, eb = synth.make_graph(seed=0, **cfg)
    deg = synth.degrees(cfg['n_users'], cfg['n_biz'], eu, eb)
    pcfg = dict(cfg)
    pcfg['n_pairs'] = per_gpu
    # shard `rank` of the job, drawn exactly like the N=1 workload (rank 0's shard IS the N=1 workload)
    pu, pv = synth.make_pairs(edge_u=eu, edge_b=eb, seed=1 + rank, deg=deg, **pcfg)

    ug = a.cpu_user_groups or 600 * cores
    bg = a.cpu_biz_groups or 250 * cores

    if a.impl == 'reference':
        if rank != 0:
            return
        t0 = time.perf_counter()
        vals = []
        for _ in range(a.steps):
            rate, sample, sides = cpu_reference_all_cores(cfg, eu, eb, pu, pv, ug, bg, cores)
            vals.append(rate)
        rate = statistics.median(vals)
        try:
            sides.update(cpu_c1_legs())
        except Exception as exc:
            sides['c1_legs_error'] = repr(exc)
        line = {'metric': METRIC, 'value': rate, 'unit': UNIT, 'impl': 'reference',
                'n_gpus': a.gpus, 'steps': len(vals), 'warmup': 0,
                'ms_per_step': (time.perf_counter() - t0) * 1e3 / len(vals),
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'int64',
                'data': 'synthetic', 'config': config,
                'cpu_baseline': {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                                 'sample': sample, 'note': NOTE, 'sides': sides},
                'e2e': {'value': rate, 'unit': UNIT, 'h2d_bytes_per_step': 0,
                        'd2h_bytes_per_step': 0}}
        print(json.dumps(line), flush=True)
        return

    cpu_baseline, c_full = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        # single-process figure first (BASELINE.md section 2: the >=100x target is judged on it)
        sg_u = a.cpu_user_groups or 1500
        sg_b = a.cpu_biz_groups or 600
        rate, sample, sides = cpu_single_process(cfg, eu, eb, pu, pv, sg_u, sg_b)
        try:
            sides.update(cpu_c1_legs())
        except Exception as exc:
            sides['c1_legs_error'] = repr(exc)
        try:
            cs, c_full = cpu_c_port(cfg, eu, eb, pu, pv, cores)
            sides.update(cs)
        except Exception as exc:   # the C oracle is context and checker, never the headline
            sides['c_port_error'] = repr(exc)
        sides['all_core_python'] = 'see the --impl reference line of the same round (Oracle A on every core)'
        cpu_baseline = {'value': rate, 'unit': UNIT, 'cores': 1, 'kind': 'port', 'host_cores': cores,
                        'sample': sample, 'note': NOTE, 'sides': sides}

    import torch
    import torch.distributed as dist
    graph, roofline, _lib, dmod = pkg('graph'), pkg('roofline'), pkg('_lib'), pkg('dist')
    _lib.load()   # fails loudly when the CUDA extension is missing
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    t0 = time.perf_counter()
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, device=local_rank, build='host')
    build_host_s = time.perf_counter() - t0
    # SURVEY section 8f rank 1: the same graph built on the device (edge arrays already in HBM)
    deu, deb = torch.from_numpy(eu).to(dev), torch.from_numpy(eb).to(dev)
    graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], deu, deb, device=local_rank,
                         build='device').close()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Gd = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], deu, deb, device=local_rank,
                              build='device')
    build_device_s = time.perf_counter() - t0
    Gd.close()
    del deu, deb

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- the job's pair list.  N=1: this rank's shard.  N>1: all shards, concatenated, re-cut.
    n_total = per_gpu * world
    window, bounds, lo = None, None, 0
    if world > 1:
        shard_u = torch.from_numpy(pu).to(dev)
        shard_b = torch.from_numpy(pv).to(dev)
        all_u = torch.empty(n_total, dtype=torch.int32, device=dev)
        all_b = torch.empty(n_total, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(all_u, shard_u)
        dist.all_gather_into_tensor(all_b, shard_b)
        pu_all, pv_all = all_u.cpu().numpy(), all_b.cpu().numpy()
        del shard_u, shard_b
        cost = dmod.pair_costs(pu_all, pv_all, deg[0], deg[1])
        bounds = dmod.shard_bounds(pu_all, world, cost)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        d_u, d_b = all_u[lo:hi].clone(), all_b[lo:hi].clone()
        pu, pv = pu_all[lo:hi], pv_all[lo:hi]              # this rank's slice from here on
        if rank != 0:
            del all_u, all_b
        window = dmod.ResultWindow(G, n_total, columns=dmod.REFERENCE_COLUMNS, dst=0,
                                   derived=tuple(a.derive.split(',')) if a.derive else None)
        if rank == 0:
            window.attach_pairs(all_u, all_b, (lo, hi))
    else:
        d_u = torch.from_numpy(pu).to(dev)
        d_b = torch.from_numpy(pv).to(dev)
    n = int(d_u.numel())
    outs = None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    mid_event = None      # set while diagnosing: recorded after this rank's own kernels, before the wait

    def step(concurrent=False, local=False):
        # the public device-resident call: both sides + pa, one side after the other on one
        # stream, so that the per-kernel event times below are those of the kernels alone
        nonlocal outs, mid_event
        if window is not None and not local:
            # peers store their rows into rank 0's window; rank 0 derives what the window's
            # `derived` names (default: pa, under its own scoring; nothing after the rows have landed)
            dmod.score_into_window(G, d_u, d_b, window, lo)
            if mid_event is not None:
                mid_event.record()
            dmod.rows_landed(G)
            if rank == 0:
                window.derive()        # whatever is left to derive for the peers' rows (default: nothing)
        else:
            outs = G.score_pairs(d_u, d_b, out=outs, concurrent=concurrent)

    def timed(reps, **kw):
        """Sum of per-step CUDA-event times of this rank, and the per-kernel stats."""
        tot, st_u, st_b = 0.0, [], []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(**kw)
            e1.record()
            e1.synchronize()
            tot += e0.elapsed_time(e1)
            st_u.append(G.score_stats(_lib.SIDE_USER))
            st_b.append(G.score_stats(_lib.SIDE_BUSINESS))
        return tot, st_u, st_b

    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(a.warmup):
        flush.zero_()
        step()
    barrier()
    if sampler:
        sampler.wait_first()
    barrier()
    t_wall0 = time.perf_counter()
    total_ms, st_u, st_b = timed(a.steps)
    barrier()                              # N>1: every rank's rows are on rank 0 from here on
    t_wall1 = time.perf_counter()
    clocks = sampler.window(t_wall0, t_wall1) if sampler else None
    if a.dump_outputs and rank == 0:
        # now: the comparison arms below reuse these buffers
        dump_outputs(a.dump_outputs, window.tensors() if window is not None else outs,
                     dump_rows(n_total))
    ms_per_step = reduce_max(total_ms) / a.steps
    value = n_total / (ms_per_step * 1e-3)
    wall_ms_per_step = reduce_max((t_wall1 - t_wall0) * 1e3) / a.steps
    launches = sum(s['kernel_launches'] for s in st_u + st_b)
    score_ms_u = [s['score_ms'] for s in st_u]
    score_ms_b = [s['score_ms'] for s in st_b]
    light_ms_u = [s['light_ms'] for s in st_u]
    light_ms_b = [s['light_ms'] for s in st_b]
    group_ms = [x['group_ms'] + y['group_ms'] for x, y in zip(st_u, st_b)]
    su, sb = st_u[-1], st_b[-1]

    concurrent_sides, multi = None, None
    reps = max(3, min(a.steps, 10))
    if world == 1 and not a.quick:
        # ---- supplementary: the same call with the two sides on two streams (grids overlap)
        for _ in range(6):          # the two-stream pattern grows the stream-ordered pool first
            step(concurrent=True)
        barrier()
        c_ms, _, _ = timed(reps, concurrent=True)
        c_ms /= reps
        concurrent_sides = {'ms_per_step': c_ms, 'value': n_total / (c_ms * 1e-3), 'unit': UNIT,
                            'steps': reps,
                            'what': 'score_pairs(concurrent=True): business side on a second stream'}
    elif world > 1 and a.quick:
        bpp = window.bytes_per_pair()
        multi = {'bytes_per_pair_over_nvlink': bpp, 'slice_pairs': [int(bounds[r + 1] - bounds[r]) for r in range(world)],
                 'fused_window': {'ms_per_step': ms_per_step, 'value': value, 'unit': UNIT,
                                  'wall_ms_per_step_with_barriers': wall_ms_per_step}}
        if rank == 0:
            cols = window.tensors()
            try:
                from oracle import c_oracle
                idx = np.arange(0, n_total, max(1, n_total // 40_000))
                want = c_oracle.score_pair_arrays_parallel(cfg['n_users'], cfg['n_biz'], eu, eb,
                                                           pu_all[idx], pv_all[idx], threads=min(cores, 4))
                tidx = torch.from_numpy(idx).to(dev)
                chk = compare_with_oracle({k: cols[k][tidx].cpu().numpy() for k in cols}, want)
                chk['what'] = ('strided sample over the whole %d-pair list (rows of every rank) vs the C '
                               'oracle' % n_total)
                multi['oracle_check'] = chk
            except Exception as exc:
                multi['oracle_check'] = {'error': repr(exc)}
    elif world > 1:
        # ---- the two comparison arms: scoring into local memory, and local scoring + NCCL gather
        for _ in range(2):
            step(local=True)
        barrier()
        l_ms, _, _ = timed(reps, local=True)
        barrier()
        l_ms_own = l_ms / reps
        l_ms = reduce_max(l_ms) / reps
        counts = [int(bounds[r + 1] - bounds[r]) for r in range(world)]
        keep = {k: outs[k] for k in dmod.REFERENCE_COLUMNS}
        full = None
        if rank == 0:
            full = {k: torch.empty(n_total, dtype=keep[k].dtype, device=dev) for k in keep}
        for _ in range(2):
            dmod.gather_results(keep, counts, dst=0, out=full)
        barrier()
        g_tot = 0.0
        for _ in range(reps):
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            dmod.gather_results(keep, counts, dst=0, out=full)
            g1.record()
            g1.synchronize()
            g_tot += g0.elapsed_time(g1)
        barrier()
        g_ms = reduce_max(g_tot) / reps
        # diagnosis: how long each rank's OWN kernels take when they store into the window (before
        # it waits for the others), per rank
        own_ms = []
        for _ in range(reps):
            flush.zero_()
            e0 = torch.cuda.Event(enable_timing=True)
            mid_event = torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            torch.cuda.synchronize()
            own_ms.append(e0.elapsed_time(mid_event))
        mid_event = None
        barrier()
        mine = torch.tensor([statistics.mean(own_ms), l_ms_own], dtype=torch.float64, device=dev)
        per_rank = [torch.zeros(2, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(per_rank, mine)
        bpp = window.bytes_per_pair()
        multi = {'bytes_per_pair_over_nvlink': bpp,
                 'per_rank_own_kernels_ms': {'into_window': [float(t[0]) for t in per_rank],
                                             'into_local_memory': [float(t[1]) for t in per_rank]},
                 'bytes_into_rank0_per_step': bpp * (n_total - n if rank == 0 else 0),
                 'slice_pairs': counts,
                 'fused_window': {'ms_per_step': ms_per_step, 'value': value, 'unit': UNIT,
                                  'wall_ms_per_step_with_barriers': wall_ms_per_step,
                                  'what': 'every rank\'s kernels store its rows into rank 0\'s peer-mapped window '
                                          '(the business side by copy engine under the user-side kernels); '
                                          'rank 0 derives %s (this is the line\'s `value`)' % ', '.join(window.derived)},
                 'scoring_only': {'ms_per_step': l_ms, 'value': n_total / (l_ms * 1e-3), 'unit': UNIT,
                                  'what': 'same slices scored into local memory, nothing gathered'},
                 'nccl_gather': {'gather_ms': g_ms, 'ms_per_step': l_ms + g_ms,
                                 'value': n_total / ((l_ms + g_ms) * 1e-3), 'unit': UNIT,
                                 'what': 'local scoring, then dist.gather_results: one grouped batch '
                                         'of NCCL send/recv of the seven columns into rank 0'}}
        # ---- every rank's rows, as they sit on rank 0, against the unsharded call and the oracle
        if rank == 0:
            cols = window.tensors()
            whole = G.score_pairs(all_u, all_b)
            torch.cuda.synchronize()
            multi['all_rows_match_unsharded_call'] = bool(all(torch.equal(cols[k], whole[k]) for k in cols))
            multi['nccl_gather_rows_match'] = bool(all(torch.equal(cols[k], full[k]) for k in cols))
            del whole
            try:
                from oracle import c_oracle
                idx = np.arange(0, n_total, max(1, n_total // 200_000))
                want = c_oracle.score_pair_arrays_parallel(cfg['n_users'], cfg['n_biz'], eu, eb,
                                                           pu_all[idx], pv_all[idx], threads=cores)
                tidx = torch.from_numpy(idx).to(dev)
                got = {k: cols[k][tidx].cpu().numpy() for k in cols}
                chk = compare_with_oracle(got, want)
                chk['what'] = ('strided sample over the whole %d-pair list (rows of every rank) vs the C '
                               'oracle' % n_total)
                multi['oracle_check'] = chk
            except Exception as exc:
                multi['oracle_check'] = {'error': repr(exc)}
            del full
        outs = None

    # ---- end to end through the host-buffer API (the seven reference outputs: 48 B per pair)
    e2e, host = None, None
    if a.quick:
        # no host-buffer leg: the columns the roofline / parity code needs come off the device
        if rank == 0:
            if world > 1:
                cols = window.tensors()
                host = {k: cols[k][lo:lo + n].cpu().numpy() for k in ('u_cn', 'b_cn')}
            else:
                host = {k: v.cpu().numpy() for k, v in outs.items()}
    else:
        sess = G.host_session(n)
    hu, hb = (sess.pinned_inputs(n) if not a.quick else (None, None))
    if not a.quick:
        hu[:] = pu
        hb[:] = pv
        e2e_steps = max(3, min(a.steps, 10))
        link = sess.measure_link(n) if rank == 0 else None     # (scribbles over the result buffers: first)
        for _ in range(2):
            sess.score_pinned(n)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            host = sess.score_pinned(n)
        torch.cuda.synchronize()
        e2e_s = reduce_max(time.perf_counter() - t0) / e2e_steps
        e2e = {'value': n_total / e2e_s, 'unit': UNIT, 'ms_per_step': e2e_s * 1e3,
               'h2d_bytes_per_step': sess.h2d_bytes_per_pair * n,
               'd2h_bytes_per_step': sess.d2h_bytes_per_pair * n, 'steps': e2e_steps,
               'columns': list(sess.KEYS), 'link': link,
               'api': 'BipartiteGraph.host_session().score_pinned -> one blp_score_pairs_host call '
                      '(pinned host buffers in and out, both sides + pa; per rank at N>1)'}
        del sess

    # ---- the other BASELINE.json configs, briefly (N=1: a part of C3 and of C4; N>1: C3 cut N ways)
    others = None
    if a.config == 'C2' and not a.quick and not a.no_other_configs:
        peak_o = 6650.0
        try:
            peak_o = float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))).get('hbm_gbs', 6650.0))
        except (OSError, ValueError):
            pass
        plan = [('C3', 20_000_000), ('C4', 10_000_000)] if world == 1 else [('C3', 100_000_000)]
        others = []
        for oname, opairs in plan:
            try:
                ol = other_config_line(oname, opairs, 3, rank, world, dev, cores, peak_o)
            except Exception as exc:      # never lose the headline line to a side measurement
                ol = {'config': oname, 'error': repr(exc)}
                if world > 1:
                    raise
            if rank == 0:
                others.append(ol)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except (OSError, ValueError):
            pass
        peak = float(peaks.get('hbm_gbs', 6650.0))
        ab = roofline.algorithmic_bytes(cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv,
                                        host['u_cn'], host['b_cn'])
        parity = None
        if c_full is not None:
            parity = compare_with_oracle(host, c_full)
            parity['what'] = ('ALL %d pairs of the timed workload: blp_score_pairs_host output vs the '
                              'plain-C oracle (oracle/blp_oracle.c)' % n)
        traffic, traffic_src, phase = None, None, None
        tj = _profile_json('r02_traffic.json')
        if tj and a.config == tj.get('config', 'C2') and per_gpu == cfg['n_pairs'] and world == 1:
            traffic = tj['user_side']['traffic_bytes']     # the capture is of this workload
            traffic_src = tj['source']
        pj = _profile_json('r02_phase_shares.json')
        if pj and a.config == pj.get('config', 'C2'):
            phase = pj
        ku_ms = statistics.mean(score_ms_u)
        kb_ms = statistics.mean(score_ms_b)
        bytes_u = ab['user'] + ab['pa']
        ach = bytes_u / (ku_ms * 1e-3) / 1e9
        roof = {'bound': 'hbm', 'kernel': 'user side = k_score_side (CTA per group) with '
                'k_score_light (warp per light group) beside it on the handle\'s side stream: '
                'two-hop expansion + intersection + epilogue, PA folded in; kernel_ms spans both',
                'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak,
                'peak_source': 'MEASURED_PEAKS.json hbm_gbs (of measured)' if peaks
                else 'fallback 6650 GB/s (of fallback)',
                'traffic': traffic, 'traffic_source': traffic_src,
                'algorithmic_bytes_per_launch': bytes_u,
                'kernel_ms': ku_ms,
                'k_score_light_span_ms': statistics.mean(light_ms_u),
                'work_items': {'user_side': su['n_groups'], 'user_side_warp_kernel': su['light_groups'],
                               'business_side': sb['n_groups'],
                               'business_side_warp_kernel': sb['light_groups']},
                'launch': {'ctas': su['ctas'], 'threads_per_cta': su['threads_per_cta'],
                           'smem_bytes': su['smem_bytes'], 'range_passes': su['range_passes']},
                'business_kernel': {'kernel_ms': kb_ms,
                                    'k_score_light_ms': statistics.mean(light_ms_b),
                                    'algorithmic_bytes_per_launch':
                                    ab['business'],
                                    'achieved': ab['business'] / (kb_ms * 1e-3) / 1e9},
                'grouping_ms_per_step': statistics.mean(group_ms),
                'note': 'the graph is L2-resident for C1-C4: DRAM traffic is far below the '
                        'algorithmic bytes; the kernels are latency/issue-bound, and the probe / table '
                        'paths answer hub-partner pairs without streaming the partner list, so the '
                        'algorithmic figure credits bytes the implementation does not move -- see '
                        'profiles/r02_notes.md.',
                'whole_step': {'algorithmic_bytes': ab['total'],
                               'achieved': ab['total'] / (ms_per_step * 1e-3) / 1e9},
                'bytes_breakdown': {k: ab[k] for k in ('expansion_user', 'stream_user',
                                                       'expansion_business', 'stream_business',
                                                       'pa', 'invalid')}}
        if phase:
            # SURVEY 8d: "for the intersection kernel use the per-pair terms only over K2's own
            # time".  Expansion and intersection are fused in one launch here, so K2's own time is
            # DERIVED: this run's kernel time x the intersection phase's share of the CTA kernel's
            # cycles, measured with the instrumented build of the SAME kernels (tools/phase_time.py).
            share = phase['intersection_share_of_user_side']
            t_int = ku_ms * share
            roof['intersection_phase'] = {
                'derived': True, 'share_of_kernel': share,
                'share_source': phase['source'], 'time_ms': t_int,
                'algorithmic_bytes': ab['stream_user'],
                'achieved': ab['stream_user'] / (t_int * 1e-3) / 1e9,
                'frac': ab['stream_user'] / (t_int * 1e-3) / 1e9 / peak}
        if cpu_baseline:
            fair1 = cpu_baseline['value']
            cpu_baseline['target_100x'] = {
                'vs_fair_single_process': {'device_resident': value / fair1,
                                           'e2e': e2e['value'] / fair1 if e2e else None},
                'vs_c_port_all_cores': None}
            allc = cpu_baseline['sides'].get('c_port_all_cores_pairs_per_s')
            if allc:
                cpu_baseline['target_100x']['vs_c_port_all_cores'] = {
                    'device_resident': value / allc, 'e2e': e2e['value'] / allc if e2e else None}
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps,
                'warmup': a.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None, 'dtype': 'int64', 'data': 'synthetic',
                'config': config, 'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches,
                'roofline': roof, 'cpu_baseline': cpu_baseline, 'parity_full_workload': parity,
                'multi_gpu': multi, 'concurrent_sides': concurrent_sides, 'other_configs': others,
                'graph': G.info(),
                'graph_build': {'host_builder_s': build_host_s, 'device_builder_s': build_device_s,
                                'edge_lines': int(eu.size),
                                'what': 'blp_graph_create (host arrays, first call: includes CUDA '
                                        'context creation) vs blp_graph_create_device (edges in HBM)'}}
        print(json.dumps(line), flush=True)
    if sampler:
        sampler.stop()
    if world > 1:
        barrier()
        window.close()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
