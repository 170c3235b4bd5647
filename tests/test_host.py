"""CPU tests of the host layer: C-ABI exports, error behaviour without a GPU, formats, sharding."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, pkg


def test_library_exports_every_declared_symbol(built_lib):
    header = open(os.path.join(ROOT, 'include', 'blp.h')).read()
    declared = set(re.findall(r'\b(blp_[a-z_0-9]+)\s*\(', header))
    assert {'blp_graph_create', 'blp_score_pairs', 'blp_graph_destroy', 'blp_last_error'} <= declared
    for name in declared:
        assert hasattr(built_lib, name), 'libblp.so does not export %s' % name
    assert set(pkg('_lib').EXPORTS) == declared
    assert built_lib.blp_version() >= 100


NO_DEVICE_CHECKS = r'''
import ctypes
import sys
import torch
sys.path.insert(0, sys.argv[1])
from conftest import pkg
assert not torch.cuda.is_available()
lib_mod = pkg('_lib')
lib = lib_mod.load()
n = ctypes.c_int(-1)
assert lib.blp_device_count(ctypes.byref(n)) == lib_mod.BLP_ERR_CUDA and n.value == 0
assert b'CUDA' in lib.blp_last_error()
try:
    pkg('graph').BipartiteGraph(4, 3, [0, 1], [0, 1])       # fails loudly, never computes on CPU
except RuntimeError:
    pass
else:
    raise AssertionError('BipartiteGraph was created without a CUDA device')
'''


def test_no_cpu_fallback_without_device(built_lib):
    """Run in a child process that sees no CUDA device, so that it runs on GPU machines too."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    res = subprocess.run([sys.executable, '-c', NO_DEVICE_CHECKS, os.path.join(ROOT, 'tests')], env=env,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-4000:]


def test_argument_validation_precedes_device_use(built_lib):
    lib_mod = pkg('_lib')
    h = ctypes.c_void_p()
    assert built_lib.blp_graph_create(0, 3, 0, None, None, 0, ctypes.byref(h)) == lib_mod.BLP_ERR_INVALID
    assert built_lib.blp_graph_create(4, 3, 2, None, None, 0, ctypes.byref(h)) == lib_mod.BLP_ERR_INVALID
    assert built_lib.blp_graph_destroy(None) == lib_mod.BLP_OK
    assert built_lib.blp_score_pairs(None, 0, None, None, 0, *([None] * 7)) == lib_mod.BLP_ERR_INVALID
    assert built_lib.blp_score_pairs_host(None, None, None, 0, *([None] * 9), 0, -1, 0) \
        == lib_mod.BLP_ERR_INVALID
    assert b'blp_score_pairs_host' in built_lib.blp_last_error()
    with pytest.raises(ValueError):
        lib_mod.check(lib_mod.BLP_ERR_INVALID, 'x')
    with pytest.raises(RuntimeError):
        lib_mod.check(lib_mod.BLP_ERR_CUDA, 'x')


def test_synth_is_seeded_and_well_formed():
    synth = pkg('synth')
    cfg, eu, eb, pu, pv = synth.make_config('C1')
    cfg2, eu2, eb2, pu2, pv2 = synth.make_config('C1')
    assert np.array_equal(eu, eu2) and np.array_equal(pv, pv2)
    assert eu.size == cfg['n_reviews'] and pu.size == cfg['n_pairs'] == 100_000
    assert eu.min() >= 0 and eu.max() < cfg['n_users'] and eb.max() < cfg['n_biz']
    assert np.all(np.diff(pu[pu >= 0]) >= 0)                     # grouped by user
    ok = (pu >= 0) & (pv >= 0)
    assert 50 <= (~ok).sum() <= 200                              # ~0.1 % literal-0 pairs
    key = pu[ok].astype(np.int64) * cfg['n_biz'] + pv[ok]
    assert np.unique(key).size == key.size                       # K distinct businesses per user
    # rank shards tile the example users without overlap
    parts = [synth.make_config('C1', rank=r, world=4)[3] for r in range(4)]
    assert sum(p.size for p in parts) == cfg['n_pairs']
    us = [set(p[p >= 0].tolist()) for p in parts]
    assert not (us[0] & us[1]) and not (us[2] & us[3])


def test_json_formats_round_trip(tmp_path):
    util, synth = pkg('util'), pkg('synth')
    ids_u, ids_b = synth.shared_ids(10, np.array([1, 1, -1]), np.array([0, 3, 2]))
    ex = synth.examples_dict(ids_u, ids_b)
    f = str(tmp_path / 'examples.json')
    util.write_json(ex, f)
    back = util.load_json(f)
    assert back == ex and all(isinstance(k, str) for k in back)
    assert back['1'] == {'10': 0, '13': 0}
    util.write_edge_list(str(tmp_path / 'g.txt'), [0, 5], [10, 12])
    assert open(str(tmp_path / 'g.txt')).read() == '0 10\n5 12\n'
    u, b = pkg('graph').read_edge_list(str(tmp_path / 'g.txt'))
    assert u.tolist() == [0, 5] and b.tolist() == [10, 12]


def test_columnar_sidecar_is_lossless(tmp_path):
    """JSON -> npz -> JSON reproduces the reference's score file byte for byte (types included)."""
    util = pkg('util')
    scores = {'3': {'10': 2, '11': 0.5, '12': 0}, '7': {'10': 0, '13': 1.4426950408889634},
              '9': {'11': 0.0}}
    fj, fn, fb = (str(tmp_path / n) for n in ('s.json', 's.npz', 'back.json'))
    util.write_json(scores, fj)
    util.json_to_npz(fj, fn)
    util.npz_to_json(fn, fb)
    assert open(fb).read() == open(fj).read()
    back = util.load_json(fb)
    assert isinstance(back['3']['12'], int) and isinstance(back['9']['11'], float)
    u, b, v, im = util.dict_to_columns(scores)
    assert u.tolist() == [3, 3, 3, 7, 7, 9] and im.tolist() == [True, False, True, True, False, False]


def test_set_level_functions_keep_reference_meaning():
    sim = pkg('similarity')

    class G(object):
        def GetNI(self, i):
            class NI(object):
                def GetDeg(_self):
                    return {1: 1, 2: 2, 5: 2}[i]
            return NI()

    a, b = {1, 2, 5}, {2, 3, 5}
    assert sim.common_neighbors(a, b) == 2
    assert sim.jaccard(a, b) == 0.5
    assert sim.adamic_adar(a, b, G()) == pytest.approx(2.8853900817779268, rel=1e-15)
    assert sim.adamic_adar({1}, {1}, G()) == 0 and isinstance(sim.adamic_adar({1}, {1}, G()), int)
    assert sim.preferential_attachment({10, 11}, {2, 3, 5}) == 6
    with pytest.raises(ZeroDivisionError):
        sim.jaccard(set(), set())


def test_id_lookup():
    graph = pkg('graph')
    table = np.array([3, 7, 9, 40], dtype=np.int64)
    got = graph.BipartiteGraph._lookup(table, [7, 8, 40, 41, -1, 3])
    assert got.tolist() == [1, -1, 3, -1, -1, 0]


def test_shard_bounds_are_user_aligned_and_balanced():
    dist = pkg('dist')
    rng = np.random.default_rng(0)
    pu = np.repeat(np.arange(200), rng.integers(1, 40, 200))
    cost = rng.random(pu.size) * 10
    for world in (1, 2, 3, 8):
        b = dist.shard_bounds(pu, world, cost)
        assert b[0] == 0 and b[-1] == pu.size and np.all(np.diff(b) >= 0) and b.size == world + 1
        for cut in b[1:-1]:
            assert cut == 0 or cut == pu.size or pu[cut] != pu[cut - 1]     # never inside a user
        per = [cost[b[r]:b[r + 1]].sum() for r in range(world)]
        assert max(per) <= cost.sum() / world + 2 * 40 * 10
    assert dist.shard_bounds(np.zeros(0, np.int32), 4).tolist() == [0, 0, 0, 0, 0]


def test_algorithmic_bytes_on_known_answer():
    import json
    roofline = pkg('roofline')
    ka = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'known_answer.json')))
    lines = np.array(ka['graph_lines'])
    pu = np.array([p['u'] if p['u'] < 6 else -1 for p in ka['pairs']])
    pv = np.array([p['v'] - 10 if 10 <= p['v'] < 14 else -1 for p in ka['pairs']])
    u_cn = [p['u_cn'] for p in ka['pairs']]
    b_cn = [p['b_cn'] for p in ka['pairs']]
    ab = roofline.algorithmic_bytes(6, 4, lines[:, 0], lines[:, 1] - 10, pu, pv, u_cn, b_cn)
    # user side by hand: distinct users {0,1,2,3,4}; deg 2,1,2,2,1; expansion 5,3,5,5,2
    assert ab['expansion_user'] == 4 * ((2 + 1 + 2 + 2 + 1) + (5 + 3 + 5 + 5 + 2))
    # 8 in-graph pairs: 32 B each + 4*deg(v) + 8*u_cn
    degv = [3, 2, 2, 3, 3, 3, 3, 3]
    assert ab['stream_user'] == 32 * 8 + 4 * sum(degv) + 8 * sum(u_cn[:8])
    assert ab['invalid'] == 64 and ab['pa'] == 80
    assert ab['total'] == ab['user'] + ab['business'] + ab['pa']


def test_result_window_layout():
    """The memory plan of the multi-GPU result window (pure host logic of dist.ResultWindow)."""
    d = pkg('dist')
    n = 1000
    ref = d.window_layout(n)                                   # the seven reference columns, pa derived
    assert ref['columns'] == d.REFERENCE_COLUMNS and ref['derived'] == ('pa',)
    assert ref['allocated'] == d.REFERENCE_COLUMNS             # nothing extra is needed to derive pa
    assert 'pa' not in ref['wire'] and ref['wire_bytes_per_pair'] == 40
    # 32 bytes on the wire: jaccard derived too, which needs cn and union in the window
    c32 = d.window_layout(n, derived=d.DERIVED_COLUMNS)
    assert set(c32['wire']) == set(d.WIRE_COLUMNS) and c32['wire_bytes_per_pair'] == 32
    assert {'u_union', 'b_union'} <= set(c32['allocated']) and 'u_union' not in c32['columns']
    # everything stored by the kernels
    full = d.window_layout(n, columns=d.ALL_COLUMNS, compact=False)
    assert full['derived'] == () and full['wire_bytes_per_pair'] == 56
    # a column that is not asked for is neither allocated nor derived
    few = d.window_layout(n, columns=('u_cn', 'b_adamic'))
    assert few['derived'] == () and few['allocated'] == ('u_cn', 'b_adamic') and few['wire_bytes_per_pair'] == 12
    for plan in (ref, c32, full, few):
        spans = sorted((plan['offsets'][c], {'cn': 4, 'union': 4}.get(c.split('_')[-1], 8) * n) for c in plan['allocated'])
        assert all(o % 256 == 0 for o, _ in spans)
        assert all(a + la <= b for (a, la), (b, _) in zip(spans, spans[1:]))      # columns do not overlap
        assert spans[-1][0] + spans[-1][1] <= plan['nbytes']
    with pytest.raises(ValueError):
        d.window_layout(n, columns=('u_cn', 'nope'))
    with pytest.raises(ValueError):
        d.window_layout(n, derived=('u_cn',))
