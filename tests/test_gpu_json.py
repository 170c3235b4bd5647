"""The JSON ends of similarity.main on the device (csrc/blp_json.cu): the score-file writer against
json.dumps of the dict similarity._emit builds, the examples.json reader against json.load +
similarity._flatten, and main's device path against the host path (util.load_json + users +
business), byte for byte."""
import json
import math
import os
import sys

import numpy as np
import pytest

from conftest import pkg

pytestmark = pytest.mark.gpu

# method -> (column, kind) as main writes it; 'nope' is an unknown method name (zeros only)
METHOD_OF_KIND = {'cn': 'common_neighbors', 'pa': 'preferential_attachment', 'jaccard': 'jaccard',
                  'adamic': 'adamic_adar'}
ALL_METHODS = ['common_neighbors', 'jaccard', 'adamic_adar', 'preferential_attachment', 'nope']


@pytest.fixture(scope='module')
def env(built_lib):
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    return torch, pkg('similarity'), pkg('util'), pkg('_lib')


# ------------------------------------------------------------------------------------ writer
def write_both(env, tmp_path, uids, counts, biz, in_graph, vals, col, chunk_bytes=None, tag='doc'):
    """(device bytes, _emit bytes) of one score file; col None = zeros only."""
    torch, sim, util, _lib = env
    uids = np.asarray(uids, dtype=np.int64)
    counts = np.asarray(counts, dtype=np.int64)
    biz = np.asarray(biz, dtype=np.int64)
    in_graph = np.asarray(in_graph, dtype=bool)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    d = torch.device('cuda', 0)
    dv = None if col is None else torch.from_numpy(np.ascontiguousarray(vals)).to(d)
    f_dev, f_ref = str(tmp_path / (tag + '_dev.json')), str(tmp_path / (tag + '_ref.json'))
    kw = {} if chunk_bytes is None else {'chunk_bytes': chunk_bytes}
    util.write_scores_json_device(f_dev, torch.from_numpy(off).to(d), torch.from_numpy(uids).to(d),
                                  torch.from_numpy(biz).to(d), torch.from_numpy(in_graph).to(d), dv,
                                  None if col is None else sim._KIND[col], **kw)
    keys_u = [str(u) for u in np.repeat(uids, counts).tolist()]
    keys_b = [str(b) for b in biz.tolist()]
    method = 'nope' if col is None else METHOD_OF_KIND[col]
    host = {} if col is None else {col: np.asarray(vals)}
    sim._emit(None, keys_u, keys_b, host, in_graph, [method], [f_ref])
    return open(f_dev, 'rb').read(), open(f_ref, 'rb').read()


def value_classes():
    """The doubles tests/test_json_format.py checks on the host, as one array."""
    uni = np.concatenate([np.full(u, u) for u in range(1, 1001)]).astype(np.float64)
    cn = np.concatenate([np.arange(1, u + 1) for u in range(1, 1001)]).astype(np.float64)
    bits = np.random.default_rng(20181).integers(0, 2 ** 64, size=1_000_000, dtype=np.uint64).view(np.float64)
    p10 = np.array([float('1e%d' % k) for k in range(-323, 309)])
    with np.errstate(over='ignore'):
        p10 = np.concatenate([np.nextafter(p10, -np.inf), p10, np.nextafter(p10, np.inf)])
    special = [1e-4, 1e-5, 1e16, 9999999999999998.0, 1e23, 5e-324, sys.float_info.min,
               sys.float_info.max, 2.0 ** 53, 2.0 ** 53 + 2, 2.0 ** 53 - 1, -0.0, 0.0,
               float('nan'), float('inf'), float('-inf')]
    aa = np.arange(0, 1 << 18, dtype=np.float64) / 2.0 ** 31
    v = np.concatenate([cn / uni, bits[np.isfinite(bits)], [math.ldexp(1.0, e) for e in range(-1074, 1024)],
                        p10, -p10, special, aa])
    return v


def test_writer_value_classes_one_and_many_users(env, tmp_path):
    v = value_classes()
    n = v.size
    ig = np.ones(n, dtype=bool)
    a, b = write_both(env, tmp_path, [42], [n], np.arange(n), ig, v, 'jaccard', tag='one')
    assert a == b
    rng = np.random.default_rng(5)
    counts = rng.integers(1, 70, size=n // 20)
    counts = counts[np.cumsum(counts) <= n]
    counts = np.append(counts, n - counts.sum())
    uids = rng.permutation(np.arange(counts.size, dtype=np.int64) * 7919 - 10 ** 9)
    a, b = write_both(env, tmp_path, uids, counts, np.arange(n) % 100_003 + 10 ** 17, ig, v, 'adamic', tag='many')
    assert a == b


def test_writer_kinds_masks_ids_and_chunks(env, tmp_path):
    rng = np.random.default_rng(11)
    n_users = 2000
    counts = rng.integers(0, 40, size=n_users)
    counts[:3] = 0                                   # users without pairs: absent
    n = int(counts.sum())
    i64 = np.iinfo(np.int64)
    uids = rng.choice(np.arange(-10 ** 6, 10 ** 6), size=n_users, replace=False).astype(np.int64)
    uids[3], uids[4], uids[5] = i64.min, i64.max, -1
    biz = np.concatenate([rng.choice(10 ** 6, size=c, replace=False) for c in counts]).astype(np.int64)
    biz[:4] = [i64.min, i64.max, -5, -(10 ** 18)]     # outside the random range: no duplicate keys
    i32 = np.iinfo(np.int32)
    cols = {
        'cn': rng.integers(i32.min, i32.max, size=n, dtype=np.int32),
        'pa': rng.integers(i64.min, i64.max, size=n, dtype=np.int64),
        'jaccard': rng.random(n) * (rng.random(n) < 0.8),
        'adamic': np.where(rng.random(n) < 0.3, 0.0, rng.random(n) * 5),
    }
    cols['cn'][:2] = [i32.min, i32.max]
    cols['pa'][:2] = [i64.min, i64.max]
    masks = {'all': np.ones(n, bool), 'none': np.zeros(n, bool), 'mixed': rng.random(n) < 0.7}
    for mname, ig in masks.items():
        for col in list(cols) + [None]:
            a, b = write_both(env, tmp_path, uids, counts, biz, ig, cols.get(col), col)
            assert a == b, (mname, col)
    # zeros only with every pair in the graph: every user is skipped
    a, b = write_both(env, tmp_path, uids, counts, biz, masks['all'], None, None)
    assert a == b == b'{}'
    # no users at all
    a, b = write_both(env, tmp_path, [], [], [], [], np.zeros(0), 'jaccard')
    assert a == b == b'{}'
    # chunks of ~1 KB, cut at user boundaries, give the same document as one chunk
    a, b = write_both(env, tmp_path, uids, counts, biz, masks['mixed'], cols['jaccard'], 'jaccard',
                      chunk_bytes=1024)
    whole, _ = write_both(env, tmp_path, uids, counts, biz, masks['mixed'], cols['jaccard'], 'jaccard',
                          chunk_bytes=1 << 30)
    assert a == b == whole


# ------------------------------------------------------------------------------------ reader
def check_reader(env, path):
    torch, sim, util, _lib = env
    ex = util.load_json(path)
    got = util.read_examples_device(path, 0)
    assert got is not None, path
    user_off, user_ids, biz_ids, labels = (t.cpu().numpy() for t in got)
    keys_u, keys_b, ids_u, ids_b = sim._flatten(ex)
    assert user_ids.tolist() == [int(u) for u in ex]
    assert np.diff(user_off).tolist() == [len(ex[u]) for u in ex]
    assert np.array_equal(np.repeat(user_ids, np.diff(user_off)), ids_u)
    assert np.array_equal(biz_ids, ids_b)
    assert labels.tolist() == [ex[u][b] for u, b in zip(keys_u, keys_b)]


def examples_doc(config, n_pairs, seed=3):
    synth = pkg('synth')
    cfg, eu, eb, pu, pv = synth.make_config(config, n_pairs=n_pairs)
    ids_eu, ids_eb = synth.shared_ids(cfg['n_users'], eu, eb)
    ids_pu, ids_pv = synth.shared_ids(cfg['n_users'], pu, pv)
    labels = np.random.default_rng(seed).integers(0, 2, size=pu.size)
    ex = {}
    for u, b, y in zip(ids_pu.tolist(), ids_pv.tolist(), labels.tolist()):
        ex.setdefault(str(u), {})[str(b)] = y
    return ex, ids_eu, ids_eb


@pytest.fixture(scope='module')
def c1(tmp_path_factory):
    return examples_doc('C1', None) + (tmp_path_factory.mktemp('c1'),)


@pytest.fixture(scope='module')
def c2(tmp_path_factory):
    return examples_doc('C2', 1_000_000) + (tmp_path_factory.mktemp('c2'),)


def test_reader_c1_c2_and_whitespace_variants(env, c1, c2, tmp_path):
    for ex, _, _, d in (c1, c2):
        p = str(d / 'examples.json')
        with open(p, 'w') as fh:
            fh.write(json.dumps(ex))
        check_reader(env, p)
    ex = c1[0]
    small = {u: ex[u] for u in list(ex)[:300]}
    small['-12'] = {'-999999999999999999': -2147483648, '0': 2147483647, '5': -0}
    texts = [json.dumps(small, indent=2), json.dumps(small, separators=(',', ':')),
             json.dumps(small).replace(': ', ':\t').replace(', ', ' ,\r\n'),
             ' \n{}\r\n', '{"5": {}}', '{"5": {}, "6": {"1": 1}, "7": {}}', '{ }']
    for i, t in enumerate(texts):
        p = str(tmp_path / ('v%d.json' % i))
        with open(p, 'w', newline='') as fh:
            fh.write(t)
        check_reader(env, p)


UNSUPPORTED = [
    '{"1": {"2": 0}, "1": {"3": 1}}',        # duplicate user
    '{"1": {"2": 0, "3": 1, "2": 1}}',        # duplicate business of one user
    '{"007": {"2": 0}}', '{"1": {"007": 0}}', '{"+7": {"2": 0}}', '{" 7": {"2": 0}}',
    '{"-0": {"2": 0}}', '{"1": {"-0": 0}}', '{"\\u0037": {"2": 0}}', '{"": {"2": 0}}',
    '{"1234567890123456789": {"2": 0}}',    # 19 digits
    '{"1": {"2": 0.5}}', '{"1": {"2": 1e3}}', '{"1": {"2": true}}', '{"1": {"2": null}}',
    '{"1": {"2": "0"}}', '{"1": {"2": 2147483648}}', '{"1": {"2": 01}}', '{"1": {"2": -}}',
    '{"1": {"2": {"3": 0}}}', '{"1": 5}', '{"1": [2]}', '[]',
    '{"1": {"2": 0}', '{"1": {"2": 0}} x', '{}{}', '{"1": {"2": 0},}', '{"1": {"2" 0}}',
    '\ufeff{"1": {"2": 0}}', '', '   ', '{"1": {"2": 0}}\x00',
]


def run_main(env, ex_path, graph_path, out_dir, host):
    """The files main writes (or the exception type it raises); host=True runs the host path."""
    torch, sim, util, _lib = env
    names = ['u_' + m for m in ALL_METHODS] + ['b_' + m for m in ALL_METHODS]
    paths = [str(out_dir / (n + '.json')) for n in names]
    try:
        if host:
            ex = util.load_json(ex_path)
            G = sim.LoadEdgeList(sim.PUNGraph, graph_path, 0, 1, device=0)
            sim.users(ex, G, ALL_METHODS, paths[:5])
            sim.business(ex, G, ALL_METHODS, paths[5:])
        else:
            sim.main(ex_path, graph_path, ALL_METHODS, paths[:5], ALL_METHODS, paths[5:], device=0)
    except Exception as e:      # noqa: BLE001 -- the type is what is compared
        return type(e)
    return [open(p, 'rb').read() for p in paths]


def test_reader_rejects_what_is_outside_its_grammar_and_main_falls_back(env, tmp_path):
    torch, sim, util, _lib = env
    g = str(tmp_path / 'graph.txt')
    with open(g, 'w') as fh:
        fh.write('1 2\n7 3\n7 2\n1 4\n')
    for i, t in enumerate(UNSUPPORTED):
        p = str(tmp_path / ('bad%d.json' % i))
        with open(p, 'wb') as fh:
            fh.write(t.encode('utf-8'))
        assert util.read_examples_device(p, 0) is None, t
        (tmp_path / ('d%d' % i)).mkdir()
        (tmp_path / ('h%d' % i)).mkdir()
        got = run_main(env, p, g, tmp_path / ('d%d' % i), host=False)
        want = run_main(env, p, g, tmp_path / ('h%d' % i), host=True)
        assert got == want, t


# ------------------------------------------------------------------------------------ main
def compare_main(env, doc, methods, bugs, sidecar):
    torch, sim, util, _lib = env
    ex, ids_eu, ids_eb, d = doc
    ep, gp = str(d / 'examples.json'), str(d / 'graph.txt')
    if not os.path.exists(gp):
        util.write_edge_list(gp, ids_eu, ids_eb)
    with open(ep, 'w') as fh:
        fh.write(json.dumps(ex))
    host_ex = util.load_json(ep)
    for bug in bugs:
        mine = [str(d / ('%s_%s_dev%d.json' % (s, m, bug))) for s in 'ub' for m in methods]
        ref = [str(d / ('%s_%s_host%d.json' % (s, m, bug))) for s in 'ub' for m in methods]
        k = len(methods)
        G = sim.main(ep, gp, methods, mine[:k], methods, mine[k:], device=0, reproduce_reference_bug=bug,
                     sidecar=sidecar)
        sim.users(host_ex, G, methods, ref[:k], sidecar=sidecar)
        sim.business(host_ex, G, methods, ref[k:], reproduce_reference_bug=bug, sidecar=sidecar)
        for a, b in zip(mine, ref):
            assert open(a, 'rb').read() == open(b, 'rb').read(), (a, bug)
            if sidecar:
                za, zb = np.load(a[:-5] + '.npz'), np.load(b[:-5] + '.npz')
                for key in ('u', 'b', 'v', 'int_mask'):
                    assert za[key].dtype == zb[key].dtype, (a, key)
                    assert np.array_equal(za[key], zb[key]), (a, key)


def test_main_device_path_c1_matches_host_path(env, c1):
    compare_main(env, c1, ALL_METHODS, (False, True), sidecar=True)


def test_main_device_path_c2_sample_matches_host_path(env, c2):
    compare_main(env, c2, ALL_METHODS, (False,), sidecar=False)
    compare_main(env, c2, ['adamic_adar'], (True,), sidecar=False)
