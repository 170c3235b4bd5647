"""More GPU parity: golden fixtures, file-level drop-in, C2-sized sample, sharding, stress shapes."""
import json
import os

import numpy as np
import pytest

from conftest import ROOT, pkg
from test_gpu_parity import AA_KEYS, INT_KEYS, JAC_KEYS, check_against, mods  # noqa: F401

pytestmark = pytest.mark.gpu


def test_golden_cases(mods):
    graph, synth = mods
    cases = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'cases.json')))['cases']
    for c in cases:
        G = graph.BipartiteGraph(c['n_users'], c['n_biz'], c['edge_u'], c['edge_b'])
        got = G.score_pairs_host(np.array(c['pair_u'], np.int32), np.array(c['pair_b'], np.int32))
        check_against(got, c['expect'], len(c['pair_u']))


def test_file_level_drop_in_matches_oracle_files(mods, tmp_path):
    """similarity.main(...) writes the same six JSON files the reference's main would."""
    from oracle import similarity_oracle as oa
    graph, synth = mods
    sim, util = pkg('similarity'), pkg('util')
    eu, eb = synth.make_graph(300, 60, 1200, seed=21, shift_u=1.0, shift_b=2.0)
    pu, pv = synth.make_pairs(300, 60, eu, eb, 900, k=6, seed=22, invalid_frac=0.03)
    ids_eu, ids_eb = synth.shared_ids(300, eu, eb)
    ids_pu, ids_pv = synth.shared_ids(300, pu, pv)
    util.write_edge_list(str(tmp_path / 'graph.txt'), ids_eu, ids_eb)
    util.write_json(synth.examples_dict(ids_pu, ids_pv), str(tmp_path / 'examples.json'))
    M = ['common_neighbors', 'jaccard', 'adamic_adar']
    names = ('cn', 'jaccard', 'adamic')
    for bug in (False, True):
        mine = [[str(tmp_path / ('%s_%s_mine%d.json' % (s, n, bug))) for n in names] for s in 'ub']
        ref = [[str(tmp_path / ('%s_%s_ref%d.json' % (s, n, bug))) for n in names] for s in 'ub']
        sim.main(str(tmp_path / 'examples.json'), str(tmp_path / 'graph.txt'), M, mine[0], M,
                 mine[1], reproduce_reference_bug=bug, sidecar=True)
        # the columnar sidecar converts back to the very same JSON text
        util.npz_to_json(mine[0][2][:-5] + '.npz', str(tmp_path / 'roundtrip.json'))
        assert open(str(tmp_path / 'roundtrip.json')).read() == open(mine[0][2]).read()
        oa.main(str(tmp_path / 'examples.json'), str(tmp_path / 'graph.txt'), M, ref[0], M, ref[1],
                reproduce_reference_bug=bug)
        for fm, fr in zip(mine[0] + mine[1], ref[0] + ref[1]):
            a, b = util.load_json(fm), util.load_json(fr)
            assert a.keys() == b.keys(), fm
            for u in a:
                assert a[u].keys() == b[u].keys(), (fm, u)
                for v in a[u]:
                    x, y = a[u][v], b[u][v]
                    assert type(x) is type(y), (fm, u, v, x, y)     # int 0 vs float, as the reference
                    if 'adamic' in fm:
                        assert x == pytest.approx(y, rel=1e-6), (fm, u, v)
                    else:
                        assert x == y, (fm, u, v)


def test_file_level_drop_in_matches_the_reference_files(mods, tmp_path):
    """similarity.main(...) against the six files the REFERENCE's own main() wrote for the same
    graph.txt / examples.json (tests/golden/ref_files.json, made by oracle/_ref): same key sets
    (the in-graph b_adamic entries missing, similarity.py:102), same int-vs-float types, same values."""
    sim, util = pkg('similarity'), pkg('util')
    doc = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'ref_files.json')))
    (tmp_path / 'graph.txt').write_text(doc['graph_txt'])
    util.write_json(doc['examples'], str(tmp_path / 'examples.json'))
    names = ['u_cn', 'u_jaccard', 'u_adamic', 'b_cn', 'b_jaccard', 'b_adamic']
    paths = [str(tmp_path / (n + '.json')) for n in names]
    M = ['common_neighbors', 'jaccard', 'adamic_adar']
    sim.main(str(tmp_path / 'examples.json'), str(tmp_path / 'graph.txt'), M, paths[:3], M, paths[3:],
             reproduce_reference_bug=True)
    for n, p in zip(names, paths):
        got, want = util.load_json(p), doc['score_files'][n]
        assert got.keys() == want.keys(), n
        for u in want:
            assert got[u].keys() == want[u].keys(), (n, u)
            for v in want[u]:
                x, y = got[u][v], want[u][v]
                assert type(x) is type(y), (n, u, v, x, y)
                if 'adamic' in n:
                    assert x == pytest.approx(y, rel=1e-8), (n, u, v)
                else:
                    assert x == y, (n, u, v)


def test_c2_sample_vs_c_oracle(mods):
    """BASELINE.json configs[1] graph (366k x 61k, 1.5M reviews), 300k-pair sample, C oracle."""
    from oracle import c_oracle
    graph, synth = mods
    cfg, eu, eb, pu, pv = synth.make_config('C2', n_pairs=300_000)
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    got = G.score_pairs_host(pu, pv)
    want = c_oracle.score_pair_arrays(cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv)
    check_against(got, want, pu.size)


def test_shards_equal_whole(mods):
    """Emulated ranks on one GPU: scoring user-aligned slices == scoring the whole list."""
    graph, synth = mods
    d = pkg('dist')
    cfg, eu, eb, pu, pv = synth.make_config('C1', n_pairs=40_000)
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    whole = G.score_pairs_host(pu, pv)
    du, db = synth.degrees(cfg['n_users'], cfg['n_biz'], eu, eb)
    for world in (2, 8):
        b = d.shard_bounds(pu, world, d.pair_costs(pu, pv, du, db))
        parts = [G.score_pairs_host(pu[b[r]:b[r + 1]], pv[b[r]:b[r + 1]]) for r in range(world)]
        for k in whole:
            assert np.array_equal(np.concatenate([p[k] for p in parts]), whole[k]), (world, k)


def test_hub_rows_and_big_groups(mods):
    """Lists longer than one 512-id chunk, a user with more than 256 businesses (several
    expansion tiles) and a business with more than 256 candidate pairs (several pair tiles)."""
    from oracle import c_oracle
    graph, synth = mods
    rng = np.random.default_rng(9)
    n_users, n_biz = 6000, 700
    eu = [rng.integers(0, n_users, 9000)]
    eb = [rng.integers(0, n_biz, 9000)]
    eu.append(np.arange(0, 3000))                    # business 0: hub with 3000 users (6 chunks)
    eb.append(np.zeros(3000, np.int64))
    eu.append(np.full(600, 7))                       # user 7: 600 businesses (3 expansion tiles)
    eb.append(np.arange(0, 600))
    eu, eb = np.concatenate(eu), np.concatenate(eb)
    pu = np.concatenate([rng.integers(0, n_users, 4000), np.full(700, 7), rng.integers(0, n_users, 900)])
    pv = np.concatenate([rng.integers(0, n_biz, 4000), np.arange(700), np.zeros(900, np.int64)])
    G = graph.BipartiteGraph(n_users, n_biz, eu, eb)
    got = G.score_pairs_host(pu, pv)
    want = c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu, pv)
    check_against(got, want, pu.size)


def test_host_session_matches_plain_path(mods):
    """The pinned, chunked, overlapped host pipeline returns what the simple path returns."""
    graph, synth = mods
    cfg, eu, eb, pu, pv = synth.make_config('C1', n_pairs=100_000)
    rng = np.random.default_rng(3)
    perm = rng.permutation(pu.size)                 # not grouped by user: chunks cut anywhere
    pu, pv = pu[perm], pv[perm]
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    want = G.score_pairs_host(pu, pv)
    sess = G.host_session(pu.size + 10, columns='all')
    for chunks, lead in ((1, 0), (1, 1), (4, 0), (8, 1), (8, 3), (16, 20)):
        hu, hb = sess.pinned_inputs(pu.size)
        hu[:] = pu
        hb[:] = pv
        got = sess.score_pinned(pu.size, user_chunks=chunks, lead_chunks=lead)
        for k in want:
            assert np.array_equal(got[k], want[k]), (chunks, lead, k)
    got = sess.score(pu[:777], pv[:777])
    for k in want:
        assert np.array_equal(got[k], want[k][:777]), k
    # the default session brings back the seven reference outputs only (48 B per pair)
    lean = G.host_session(pu.size)
    assert lean.d2h_bytes_per_pair == 48 and 'u_union' not in lean.KEYS
    got = lean.score(pu, pv)
    assert set(got) == set(lean.REFERENCE_KEYS)
    for k in got:
        assert np.array_equal(got[k], want[k]), k


def test_hub_bitmaps_do_not_change_results(mods, monkeypatch):
    """Hub lists OR-ed as bitmaps vs every list walked id by id: bit-identical outputs."""
    graph, synth = mods
    cfg, eu, eb, pu, pv = synth.make_config('C1', n_pairs=30_000)
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    assert G.info()['n_hub_biz'] > 0 and G.info()['n_hub_users'] > 0
    with_hubs = G.score_pairs_host(pu, pv, want_hop2=True)
    monkeypatch.setenv('BLP_HUB_MIN_DEG', '0')          # 0 disables hub selection
    G2 = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    assert G2.info()['n_hub_biz'] == 0 and G2.info()['n_hub_users'] == 0
    without = G2.score_pairs_host(pu, pv, want_hop2=True)
    for k in with_hubs:
        assert np.array_equal(with_hubs[k], without[k]), k


def test_id_range_passes_do_not_change_results(mods, monkeypatch):
    """Bitmap cut into id ranges (several passes per group) vs one pass: bit-identical.
    (BLP_RANGES is read when a handle is created.)"""
    graph, synth = mods
    lib = pkg('_lib')
    cfg, eu, eb, pu, pv = synth.make_config('C1', n_pairs=30_000)
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    one = G.score_pairs_host(pu, pv, want_hop2=True)
    assert G.score_stats(lib.SIDE_USER)['range_passes'] == 1
    for r, build in (('2', 'device'), ('5', 'device'), ('3', 'host'), ('7', 'host')):
        # a ranged side keeps its middle rows partitioned by range (either entry point), and a pass
        # walks only its segment of every list
        monkeypatch.setenv('BLP_RANGES', r)
        G2 = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, build=build)
        many = G2.score_pairs_host(pu, pv, want_hop2=True)
        assert G2.score_stats(lib.SIDE_USER)['range_passes'] == int(r)
        assert 2 <= G2.score_stats(lib.SIDE_BUSINESS)['range_passes'] <= int(r)   # 2000 bits: fewer, word-aligned ranges
        for k in one:
            assert np.array_equal(one[k], many[k]), (r, build, k)
    monkeypatch.delenv('BLP_RANGES')
    again = G.score_pairs_host(pu, pv, want_hop2=True)      # the first handle never saw the variable
    assert G.score_stats(lib.SIDE_USER)['range_passes'] == 1
    for k in one:
        assert np.array_equal(one[k], again[k]), k


def test_interleaved_handles_of_different_size(mods):
    """Two handles on one device whose bitmaps differ in size (a train and a test graph): scoring
    big, small, big again must work -- the shared-memory opt-in is per kernel and process, not
    per handle, and is only ever raised."""
    import torch
    from oracle import c_oracle
    graph, synth = mods
    big = (200_000, 3000, 300_000)
    small = (5_000, 3000, 20_000)
    built = []
    for (nu, nb, nr), seed in ((big, 31), (small, 32)):
        eu, eb = synth.make_graph(nu, nb, nr, seed=seed, shift_u=5.0, shift_b=5.0)
        pu, pv = synth.make_pairs(nu, nb, eu, eb, 8000, k=8, seed=seed + 1)
        G = graph.BipartiteGraph(nu, nb, eu, eb)
        built.append((G, nu, nb, eu, eb, pu, pv))
    prev = torch.cuda.current_device()
    for which in (0, 1, 0, 1, 0):
        G, nu, nb, eu, eb, pu, pv = built[which]
        got = G.score_pairs_host(pu, pv)
        want = c_oracle.score_pair_arrays(nu, nb, eu, eb, pu, pv)
        check_against(got, want, pu.size)
    assert torch.cuda.current_device() == prev      # entry points restore the caller's device


def test_universe_larger_than_shared_memory(mods):
    """2.5M users: the hop-2 bitmap (312 KB) exceeds one CTA's shared memory -> automatic ranges."""
    from oracle import c_oracle
    graph, synth = mods
    lib = pkg('_lib')
    n_users, n_biz = 2_500_000, 3000
    eu, eb = synth.make_graph(n_users, n_biz, 400_000, seed=5, shift_u=50.0, shift_b=5.0)
    pu, pv = synth.make_pairs(n_users, n_biz, eu, eb, 20_000, k=8, seed=6)
    want = c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu, pv)
    for build in ('device', 'host'):
        G = graph.BipartiteGraph(n_users, n_biz, eu, eb, build=build)
        got = G.score_pairs_host(pu, pv)
        assert G.score_stats(lib.SIDE_USER)['range_passes'] >= 2
        assert G.score_stats(lib.SIDE_BUSINESS)['range_passes'] == 1
        check_against(got, want, pu.size)
        G.close()


@pytest.mark.timeout(600)
def test_full_c2_properties(mods):
    """Full BASELINE.json configs[1] size (10M pairs): size-independent properties."""
    import torch
    graph, synth = mods
    lib = pkg('_lib')
    cfg, eu, eb, pu, pv = synth.make_config('C2')
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    du, dv = torch.from_numpy(pu).cuda(), torch.from_numpy(pv).cuda()
    r = G.score_pairs(du, dv, want_hop2=True)
    deg_u = torch.from_numpy(G.degrees(lib.SIDE_USER)).cuda().long()
    deg_b = torch.from_numpy(G.degrees(lib.SIDE_BUSINESS)).cuda().long()
    ok = (du >= 0) & (dv >= 0)
    ok &= (deg_u[du.clamp(min=0).long()] > 0) & (deg_b[dv.clamp(min=0).long()] > 0)
    u, v = du[ok].long(), dv[ok].long()
    # union = |hop2| + deg(partner) - cn, both sides; pa = deg(u)*deg(v)
    assert torch.equal(r['u_union'][ok].long(), r['u_hop2'][ok].long() + deg_b[v] - r['u_cn'][ok].long())
    assert torch.equal(r['b_union'][ok].long(), r['b_hop2'][ok].long() + deg_u[u] - r['b_cn'][ok].long())
    assert torch.equal(r['pa'][ok], deg_u[u] * deg_b[v])
    # jaccard == cn/union bit-exactly in fp64
    assert torch.equal(r['u_jaccard'][ok], r['u_cn'][ok].double() / r['u_union'][ok].double())
    assert torch.equal(r['b_jaccard'][ok], r['b_cn'][ok].double() / r['b_union'][ok].double())
    # bounds: 0 <= cn <= min(|hop2|, deg(partner)); aa <= cn/ln 2; aa == 0 needs cn weights 0
    assert bool((r['u_cn'][ok].long() <= torch.minimum(r['u_hop2'][ok].long(), deg_b[v])).all())
    assert bool((r['b_cn'][ok].long() <= torch.minimum(r['b_hop2'][ok].long(), deg_u[u])).all())
    assert bool((r['u_adamic'] <= r['u_cn'].double() / np.log(2.0) + 1e-9).all())
    # "no length-3 path" is seen from both sides alike when u is not adjacent to v:
    # u_cn == 0 and b_cn == 0 can differ only for existing edges
    differ = (r['u_cn'][ok] == 0) != (r['b_cn'][ok] == 0)
    assert int(differ.sum()) <= int(ok.sum()) // 100
    # pairs with an id that is not in the graph are all-zero
    for k, t in r.items():
        assert not bool(t[~ok].any()), k
    # same input twice -> bit-identical (no float atomics, order-independent accumulation)
    r2 = G.score_pairs(du, dv)
    for k in r2:
        assert torch.equal(r[k], r2[k]), k


@pytest.mark.timeout(900)
def test_full_c2_vs_c_oracle(mods):
    """The benchmarked workload itself -- BASELINE.json configs[1], all 10M pairs -- against the C
    oracle on every host core: every integer column bit-exact, jaccard bit-exact, adamic 1e-8."""
    from oracle import c_oracle
    graph, synth = mods
    cfg, eu, eb, pu, pv = synth.make_config('C2')
    assert pu.size == 10_000_000
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    got = G.score_pairs_host(pu, pv)
    want = c_oracle.score_pair_arrays_parallel(cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv)
    check_against(got, want, pu.size)


@pytest.mark.timeout(900)
@pytest.mark.parametrize('name,n_pairs,n_check', [('C3', 2_000_000, 40_000), ('C4', 1_000_000, 15_000)])
def test_large_configs_sampled_parity(mods, name, n_pairs, n_check):
    """BASELINE.json configs[2] (Yelp-2019 shape: 200 KB hop-2 bitmap, one 1024-thread CTA per SM)
    and configs[3] (heavy tail: hub businesses above 100k users) -- the full graph, a slice of the
    pair list on the GPU, a strided sample of it against the C oracle."""
    from oracle import c_oracle
    graph, synth = mods
    lib = pkg('_lib')
    cfg, eu, eb, pu, pv = synth.make_config(name, n_pairs=n_pairs)
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    info = G.info()
    if name == 'C4':
        assert info['max_biz_degree'] > 100_000            # the hubs the config is about
    got = G.score_pairs_host(pu, pv)
    assert G.score_stats(lib.SIDE_USER)['threads_per_cta'] == 1024
    idx = np.arange(0, pu.size, pu.size // n_check)[:n_check]
    want = c_oracle.score_pair_arrays(cfg['n_users'], cfg['n_biz'], eu, eb, pu[idx], pv[idx])
    check_against({k: v[idx] for k, v in got.items()}, want, idx.size)


@pytest.mark.timeout(900)
def test_c5_shape_at_half_scale_sampled_parity(mods):
    """BASELINE.json configs[4] (10M users x 1M businesses, 100M reviews) at half the node counts
    and a quarter of the reviews -- still the regime the config is about: the user-side universe
    (5M bits = 625 KB) is far beyond one CTA's shared memory, so every group takes several
    id-range passes over range-partitioned rows.  A strided sample against the C oracle.  (The
    full-scale graph takes minutes to generate on the host; its sharded run with the same check is
    recorded in profiles/r02_bench_c5_n2.json: `bench.py --config C5 --gpus 2 --quick`.)"""
    from oracle import c_oracle
    graph, synth = mods
    lib = pkg('_lib')
    cfg = dict(synth.CONFIGS['C5'])
    cfg.update(n_users=5_000_000, n_biz=500_000, n_reviews=25_000_000, n_pairs=2_000_000)
    eu, eb = synth.make_graph(seed=0, **cfg)
    pu, pv = synth.make_pairs(edge_u=eu, edge_b=eb, seed=1, **cfg)
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    got = G.score_pairs_host(pu, pv)
    assert G.score_stats(lib.SIDE_USER)['range_passes'] >= 3
    idx = np.arange(0, pu.size, pu.size // 6000)[:6000]
    want = c_oracle.score_pair_arrays_parallel(cfg['n_users'], cfg['n_biz'], eu, eb, pu[idx], pv[idx], threads=4)
    check_against({k: v[idx] for k, v in got.items()}, want, idx.size)
