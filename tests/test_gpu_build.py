"""Graph construction on the device, reached through the host-array entry point (blp_graph_create)
and the device-array one (blp_graph_create_device): against each other and against the C oracle."""
import time

import numpy as np
import pytest

from conftest import pkg
from test_gpu_parity import check_against, mods  # noqa: F401

pytestmark = pytest.mark.gpu


def same_graph(a, b):
    ia, ib = a.info(), b.info()
    for k in ('n_users', 'n_biz', 'n_edges_in', 'n_edges', 'n_users_in_graph', 'n_biz_in_graph',
              'max_user_degree', 'max_biz_degree', 'n_hub_biz', 'n_hub_users'):
        assert ia[k] == ib[k], (k, ia[k], ib[k])
    lib = pkg('_lib')
    for side in (lib.SIDE_USER, lib.SIDE_BUSINESS):
        assert np.array_equal(a.degrees(side), b.degrees(side))


@pytest.mark.parametrize('name,n_pairs', [('C1', 40_000)])
def test_device_build_scores_match_host_build(mods, name, n_pairs):
    """Host arrays (blp_graph_create) and device arrays (blp_graph_create_device) of one edge list:
    the same info, the same degrees and bit-identical scores."""
    graph, synth = mods
    cfg, eu, eb, pu, pv = synth.make_config(name, n_pairs=n_pairs)
    Gh = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, build='host')
    Gd = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, build='device')
    same_graph(Gh, Gd)
    a = Gh.score_pairs_host(pu, pv, want_hop2=True)
    b = Gd.score_pairs_host(pu, pv, want_hop2=True)
    for k in a:
        assert np.array_equal(a[k], b[k]), k            # bit-identical, adamic included


def test_device_build_small_and_odd_shapes(mods):
    from oracle import c_oracle
    graph, synth = mods
    rng = np.random.default_rng(4)
    for n_users, n_biz, n_edges in ((1, 1, 1), (5, 3, 0), (7, 300, 50), (3000, 2, 5000),
                                    (70000, 9, 40000)):
        eu = rng.integers(0, n_users, n_edges)
        eb = rng.integers(0, n_biz, n_edges)                  # heavy duplication when tiny
        pu = rng.integers(-1, n_users, 500)
        pv = rng.integers(-1, n_biz, 500)
        G = graph.BipartiteGraph(n_users, n_biz, eu, eb, build='device')
        got = G.score_pairs_host(pu, pv)
        want = c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu, pv)
        check_against(got, want, pu.size)
    lib = pkg('_lib').load()
    for build, api in (('host', b'blp_graph_create: '), ('device', b'blp_graph_create_device: ')):
        with pytest.raises(ValueError):
            graph.BipartiteGraph(4, 3, [0, 5], [0, 0], build=build)   # endpoint out of range
        assert lib.blp_last_error().startswith(api + b'edge 1 '), lib.blp_last_error()
    # the host-array entry point on the same odd shapes
    for n_users, n_biz, n_edges in ((1, 1, 1), (5, 3, 0), (3000, 2, 5000)):
        eu = rng.integers(0, n_users, n_edges)
        eb = rng.integers(0, n_biz, n_edges)
        pu = rng.integers(-1, n_users, 300)
        pv = rng.integers(-1, n_biz, 300)
        G = graph.BipartiteGraph(n_users, n_biz, eu, eb, build='host')
        check_against(G.score_pairs_host(pu, pv),
                      c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu, pv), pu.size)


def test_device_build_c2_and_timing(mods):
    """BASELINE.json configs[1] graph built on the GPU: same degrees, same scores on a sample."""
    import torch
    graph, synth = mods
    cfg, eu, eb, pu, pv = synth.make_config('C2', n_pairs=200_000)
    t0 = time.perf_counter()
    Gh = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, build='host')
    t_host = time.perf_counter() - t0
    deu, deb = torch.from_numpy(eu).cuda(), torch.from_numpy(eb).cuda()
    graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], deu, deb, build='device').close()   # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Gd = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], deu, deb, build='device')
    t_dev = time.perf_counter() - t0
    print('graph build: host %.3f s, device %.3f s' % (t_host, t_dev))
    same_graph(Gh, Gd)
    a = Gh.score_pairs_host(pu, pv)
    b = Gd.score_pairs_host(pu, pv)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_edge_list_text_parsed_on_the_device(mods, tmp_path):
    """graph.txt parsed by blp_edge_list_count / blp_edge_list_parse == the host parser, on the
    format dataset_maker.py:197 writes and on the oddities a text file can carry."""
    import torch
    graph, synth = mods
    util = pkg('util')
    # (1) a real-shaped file: one "<u> <b>\n" per review, duplicates included
    eu, eb = synth.make_graph(3000, 400, 20_000, seed=41, shift_u=2.0, shift_b=2.0)
    ids_u, ids_b = synth.shared_ids(3000, eu, eb)
    path = str(tmp_path / 'graph.txt')
    util.write_edge_list(path, ids_u, ids_b)
    hu, hb = graph.read_edge_list(path)
    du, db = graph.read_edge_list_device(path)
    assert np.array_equal(du.cpu().numpy(), hu) and np.array_equal(db.cpu().numpy(), hb)
    # (2) oddities: no trailing newline, blank lines, tabs, CRLF, leading blanks, comments, extra
    # columns, ids larger than 32 bits, a sign
    odd = ('# a comment\n\n12 34\n  7\t8  \r\n\n5000000000 6 extra columns 9\n+3 -4\n   \n99 100')
    p2 = str(tmp_path / 'odd.txt')
    open(p2, 'w').write(odd)
    c0, c1 = graph.read_edge_list_device(p2)
    assert c0.tolist() == [12, 7, 5000000000, 3, 99] and c1.tolist() == [34, 8, 6, -4, 100]
    # (3) a data line with one column is an error, not a silent zero
    p3 = str(tmp_path / 'bad.txt')
    open(p3, 'w').write('1 2\n3\n4 5\n')
    with pytest.raises(ValueError):
        graph.read_edge_list_device(p3)
    # (4) the whole route: text -> device parse -> device compaction -> device build == host route
    pu, pv = synth.make_pairs(3000, 400, eu, eb, 5000, k=5, seed=42)
    ipu, ipv = synth.shared_ids(3000, pu, pv)
    Gd = graph.BipartiteGraph.from_edge_list(path)                      # parse='device'
    Gh = graph.BipartiteGraph.from_edge_list(path, parse='host')
    assert np.array_equal(Gd.user_ids, Gh.user_ids) and np.array_equal(Gd.biz_ids, Gh.biz_ids)
    a, b = Gd.score_id_pairs(ipu, ipv), Gh.score_id_pairs(ipu, ipv)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    # an id on both sides is refused on the device route as well
    p4 = str(tmp_path / 'notbip.txt')
    open(p4, 'w').write('1 2\n2 3\n')
    with pytest.raises(ValueError):
        graph.BipartiteGraph.from_edge_list(p4)
    # an empty file has no edges
    p5 = str(tmp_path / 'empty.txt')
    open(p5, 'w').write('\n# nothing\n')
    with pytest.raises(ValueError):
        graph.BipartiteGraph.from_edge_list(p5)
