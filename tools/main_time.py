"""similarity.main end to end, by phase: the device path (examples.json parsed and every score
file formatted on the GPU, csrc/blp_json.cu) against the host path (util.load_json + users +
business) on the same files, in one process, with the byte identity of every output file.

    python tools/main_time.py [--configs C2 C3] [--out FILE]

C2 (10 M pairs) runs both paths; a larger config runs the device path only and writes its score
files one at a time, deleting each once it is measured (C3's six files are ~13 GB of text).
Inputs are synthetic (synth.make_config); examples.json is the text json.dumps writes for
{"<u>": {"<b>": label}}.  Everything is written under one temporary directory that is removed at
the end.  The GPU's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import filecmp
import importlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = 'bipartite-link-prediction_b200'
METHODS = ['common_neighbors', 'jaccard', 'adamic_adar']


def pkg(sub):
    return importlib.import_module(PKG + '.' + sub)


def gpu_identity():
    import torch
    out = {'gpu': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60)
        out['power_limit_and_max_sm_clock'] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out['power_limit_and_max_sm_clock'] = 'unavailable: %s' % e
    return out


def make_inputs(name, d):
    """graph.txt and examples.json of a config; examples in dict order (users by first pair)."""
    import torch
    synth, util, lib = pkg('synth'), pkg('util'), pkg('_lib')
    t0 = time.perf_counter()
    cfg, eu, eb, pu, pv = synth.make_config(name)
    ids_eu, ids_eb = synth.shared_ids(cfg['n_users'], eu, eb)
    ids_pu, ids_pv = synth.shared_ids(cfg['n_users'], pu, pv)
    util.write_edge_list(os.path.join(d, 'graph.txt'), ids_eu, ids_eb)
    # a missing user id is a user of its own; group the pairs as a dict would (first occurrence)
    uniq, first, inv = np.unique(ids_pu, return_index=True, return_inverse=True)
    rank = np.empty(uniq.size, dtype=np.int64)
    rank[np.argsort(first, kind='stable')] = np.arange(uniq.size)
    order = np.argsort(rank[inv], kind='stable')
    user_ids = uniq[np.argsort(rank)]
    counts = np.bincount(rank[inv], minlength=uniq.size)
    dev = torch.device('cuda', 0)
    off = torch.from_numpy(np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)).to(dev)
    labels = torch.from_numpy(np.random.default_rng(9).integers(0, 2, size=pu.size).astype(np.int32)).to(dev)
    n = int(pu.size)
    # the device writer produces exactly json.dumps' text of {"<u>": {"<b>": label}}
    util.write_scores_json_device(os.path.join(d, 'examples.json'), off, torch.from_numpy(user_ids).to(dev),
                                  torch.from_numpy(ids_pv[order]).to(dev), torch.ones(n, dtype=torch.bool, device=dev),
                                  labels, lib.JSON_INT32)
    return {'pairs': n, 'example_users': int(uniq.size),
            'examples_json_bytes': os.path.getsize(os.path.join(d, 'examples.json')),
            'input_generation_s': round(time.perf_counter() - t0, 1)}


def device_phases(d, tag, one_file_at_a_time=False):
    import torch
    sim, util, lib = pkg('similarity'), pkg('util'), pkg('_lib')
    sync = torch.cuda.synchronize
    ph, sizes = {}, {}
    ep, gp = os.path.join(d, 'examples.json'), os.path.join(d, 'graph.txt')
    sync()
    t0 = time.perf_counter()
    ex = util.read_examples_device(ep, 0)
    sync()
    ph['read_upload_parse_s'] = time.perf_counter() - t0
    assert ex is not None, 'examples.json outside the device grammar'
    t0 = time.perf_counter()
    G = sim.LoadEdgeList(sim.PUNGraph, gp, 0, 1, device=0)
    sync()
    ph['graph_s'] = time.perf_counter() - t0
    t0 = time.perf_counter()
    pairs = sim._device_pairs(G, ex)
    sync()
    ph['id_mapping_s'] = time.perf_counter() - t0
    lu, lb = pairs[4], pairs[5]
    t0 = time.perf_counter()
    res = {s: G.score_side(s, lu, lb, want_pa=True) for s in (lib.SIDE_USER, lib.SIDE_BUSINESS)}
    sync()
    ph['scoring_s'] = time.perf_counter() - t0
    stats, buffers = {}, {}
    t0 = time.perf_counter()
    for s, prefix in ((lib.SIDE_USER, 'u_'), (lib.SIDE_BUSINESS, 'b_')):
        for m in METHODS:
            f = os.path.join(d, '%s%s_%s.json' % (prefix, m, tag))
            sim._write_side(pairs, res[s], [m], [f], buffers=buffers, stats=stats)
            sizes[os.path.basename(f)] = os.path.getsize(f)
            if one_file_at_a_time:
                os.remove(f)
    ph['write_files_total_s'] = time.perf_counter() - t0
    ph['format_kernels_s'] = stats.get('format_ms', 0.0) / 1e3
    ph['d2h_copies_s'] = stats.get('d2h_ms', 0.0) / 1e3
    ph['file_writes_s'] = stats.get('write_s', 0.0)
    ph['phase_sum_s'] = sum(ph[k] for k in ('read_upload_parse_s', 'graph_s', 'id_mapping_s', 'scoring_s',
                                            'write_files_total_s'))
    del res, pairs, ex, G
    return {k: round(v, 3) for k, v in ph.items()}, sizes


def host_phases(d, tag):
    sim, util, lib = pkg('similarity'), pkg('util'), pkg('_lib')
    ph = {}
    ep, gp = os.path.join(d, 'examples.json'), os.path.join(d, 'graph.txt')
    t0 = time.perf_counter()
    examples = util.load_json(ep)
    ph['load_json_s'] = time.perf_counter() - t0
    t0 = time.perf_counter()
    G = sim.LoadEdgeList(sim.PUNGraph, gp, 0, 1, device=0)
    ph['graph_s'] = time.perf_counter() - t0
    for s, prefix in ((lib.SIDE_USER, 'u_'), (lib.SIDE_BUSINESS, 'b_')):   # users() / business()
        t0 = time.perf_counter()
        keys_u, keys_b, ids_u, ids_b = sim._flatten(examples)
        ph[prefix + 'flatten_s'] = time.perf_counter() - t0
        t0 = time.perf_counter()
        host, in_graph = sim._score_side(G, s, ids_u, ids_b)
        ph[prefix + 'score_and_copy_s'] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sim._emit(examples, keys_u, keys_b, host, in_graph, METHODS,
                  [os.path.join(d, '%s%s_%s.json' % (prefix, m, tag)) for m in METHODS])
        ph[prefix + 'dicts_dumps_writes_s'] = time.perf_counter() - t0
    ph['phase_sum_s'] = sum(ph.values())
    return {k: round(v, 3) for k, v in ph.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', nargs='+', default=['C2', 'C3'])
    ap.add_argument('--out', default=None, help='also write the JSON result here')
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'main_time.py measures on a CUDA device'
    pkg('_lib').build()
    sim = pkg('similarity')
    result = gpu_identity()
    tmp = tempfile.mkdtemp(prefix='blp_main_time_')
    try:
        result['temp_disk_free_gb'] = round(shutil.disk_usage(tmp).free / 1e9, 1)
        for name in a.configs:
            d = os.path.join(tmp, name)
            os.makedirs(d)
            r = make_inputs(name, d)
            if name == 'C2':
                r['device_path'], sizes = device_phases(d, 'dev')
                # main() itself, uninstrumented, over the same files
                paths = [os.path.join(d, '%s_%s_main.json' % (p, m)) for p in 'ub' for m in METHODS]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                sim.main(os.path.join(d, 'examples.json'), os.path.join(d, 'graph.txt'), METHODS, paths[:3],
                         METHODS, paths[3:], device=0)
                torch.cuda.synchronize()
                r['device_path']['main_s'] = round(time.perf_counter() - t0, 3)
                r['host_path'] = host_phases(d, 'host')
                same = {}
                for p in 'ub':
                    for m in METHODS:
                        f = '%s_%s_%%s.json' % (p, m)
                        h = os.path.join(d, f % 'host')
                        same[p + '_' + m] = all(filecmp.cmp(h, os.path.join(d, f % t), shallow=False)
                                                for t in ('dev', 'main'))
                r['byte_identical'] = same
                r['all_byte_identical'] = all(same.values())
                r['speedup_host_over_device_main'] = round(r['host_path']['phase_sum_s'] / r['device_path']['main_s'], 1)
            else:
                r['device_path'], sizes = device_phases(d, 'dev', one_file_at_a_time=True)
            r['score_file_bytes'] = sizes
            r['score_file_bytes_total'] = sum(sizes.values())
            result[name] = r
            shutil.rmtree(d)
            print(json.dumps({name: r}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as fh:
            json.dump(result, fh, indent=1)
    print(json.dumps(result))


if __name__ == '__main__':
    main()
