"""The business index (co-review bitmap built at graph creation, one pass over the pairs per call)
against the grouped business path it replaces and against the C oracle.

The index path must give bit-identical columns to the grouped path -- cn, union and hop2 are the
same integers, jaccard the same division, adamic the same order-independent fixed-point sum -- on
every entry point that reaches the business side.
"""
import numpy as np
import pytest

from conftest import pkg
from test_gpu_parity import check_against, mods  # noqa: F401

pytestmark = pytest.mark.gpu

ENV = ('BLP_BIZ_INDEX', 'BLP_BIZ_INDEX_MAX_MB', 'BLP_RANGES', 'BLP_HUB_MIN_DEG')


def handle(monkeypatch, graph, n_users, n_biz, eu, eb, **env):
    """A handle created under exactly `env` (the variables are read at creation)."""
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    G = graph.BipartiteGraph(n_users, n_biz, eu, eb)
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    return G


def biz_path(G):
    lib = pkg('_lib')
    return G.score_stats(lib.SIDE_BUSINESS)['path']


def index_and_grouped(monkeypatch, graph, n_users, n_biz, eu, eb, pu, pv, **env):
    """Scores with an index handle and a grouped-path handle; asserts which path each took and that
    every column, hop2 included, is bit-identical.  Returns the index handle's columns."""
    lib = pkg('_lib')
    Gi = handle(monkeypatch, graph, n_users, n_biz, eu, eb, **env)
    Gg = handle(monkeypatch, graph, n_users, n_biz, eu, eb, BLP_BIZ_INDEX=0, **env)
    assert Gi.info()['biz_index_bytes'] > 0 and Gg.info()['biz_index_bytes'] == 0
    a = Gi.score_pairs_host(pu, pv, want_hop2=True)
    if len(pu):
        assert biz_path(Gi) == lib.PATH_BIZ_INDEX
    b = Gg.score_pairs_host(pu, pv, want_hop2=True)
    if len(pu):
        assert biz_path(Gg) == lib.PATH_GROUPED
    assert set(a) == set(b)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    Gi.close()
    Gg.close()
    return a


def test_c1_full(mods, monkeypatch):
    from oracle import c_oracle
    graph, synth = mods
    cfg, eu, eb, pu, pv = synth.make_config('C1')
    got = index_and_grouped(monkeypatch, graph, cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv)
    check_against(got, c_oracle.score_pair_arrays(cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv), pu.size)


@pytest.mark.parametrize('permute', [False, True])
def test_c2_shape_reduced(mods, monkeypatch, permute):
    """C2's degree distributions at an eighth of its node and review counts; the pairs as they come
    (grouped by user) and randomly permuted."""
    from oracle import c_oracle
    graph, synth = mods
    cfg = dict(synth.CONFIGS['C2'])
    cfg.update(n_users=cfg['n_users'] // 8, n_biz=cfg['n_biz'] // 8, n_reviews=cfg['n_reviews'] // 8)
    eu, eb = synth.make_graph(seed=7, **cfg)
    pu, pv = synth.make_pairs(cfg['n_users'], cfg['n_biz'], eu, eb, 300_000, k=32, seed=8,
                              invalid_frac=0.001)
    if permute:
        perm = np.random.default_rng(9).permutation(pu.size)
        pu, pv = pu[perm].copy(), pv[perm].copy()
    got = index_and_grouped(monkeypatch, graph, cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv)
    idx = np.arange(0, pu.size, 7)
    want = c_oracle.score_pair_arrays(cfg['n_users'], cfg['n_biz'], eu, eb, pu[idx], pv[idx])
    check_against({k: v[idx] for k, v in got.items()}, want, idx.size)


def corner_graph():
    """Hand-made graph (3000 users x 2500 businesses) with the shapes the index path branches on."""
    rng = np.random.default_rng(11)
    eu, eb = [], []

    def add(u, b):
        eu.append(u)
        eb.append(b)
    for b in range(1500):                # user 0: deg 1500 (> 1024; a hub bitmap on the business side)
        add(0, b)
    for b in range(100, 140):            # user 1: deg 40 (> 32: the warp walks it)
        add(1, b)
    for u in range(100, 800):            # business 2400: a hub business with 700 reviewers
        add(u, 2400)
    add(2000, 2400)                      # user 2000's only business is the hub
    add(2500, 2450)                      # isolated star: business 2450's single reviewer, alone
    add(2501, 2451)                      # business 2451 has a single reviewer, who is also at the hub
    add(2501, 2400)
    for _ in range(12_000):              # background
        add(int(rng.integers(100, 2000)), int(rng.integers(0, 2400)))
    add(5, 7)
    add(5, 7)                            # a duplicate edge
    # user 2999 and business 2499 have degree 0
    eu, eb = np.array(eu, np.int32), np.array(eb, np.int32)
    users = [0, 1, 2, 5, 100, 101, 799, 2000, 2500, 2501, 2999]
    biz = [0, 7, 100, 139, 1499, 1500, 2400, 2450, 2451, 2499]
    pu = np.repeat(np.array(users, np.int32), len(biz))
    pv = np.tile(np.array(biz, np.int32), len(users))
    extra_u = [-1, 3000, 5, 5, 2999, 3, 0, 0, 5, 5, 2500, 2000, -7, 3000]
    extra_v = [5, 5, -1, 2500, 3, 2499, 7, 7, 7, 7, 2450, 2400, -7, 2500]   # (5, 7) is an edge
    pu = np.concatenate([pu, np.array(extra_u, np.int32), pu[::-1]])
    pv = np.concatenate([pv, np.array(extra_v, np.int32), pv[::-1]])        # duplicate pairs
    return 3000, 2500, eu, eb, pu, pv


@pytest.mark.parametrize('env', [{}, {'BLP_HUB_MIN_DEG': 0}, {'BLP_HUB_MIN_DEG': 1000}])
def test_corner_cases(mods, monkeypatch, env):
    from oracle import c_oracle
    graph, _ = mods
    n_users, n_biz, eu, eb, pu, pv = corner_graph()
    got = index_and_grouped(monkeypatch, graph, n_users, n_biz, eu, eb, pu, pv, **env)
    check_against(got, c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu, pv), pu.size)
    bad = (pu < 0) | (pu >= n_users) | (pv < 0) | (pv >= n_biz) | (pu == 2999) | (pv == 2499)
    assert not got['b_hop2'][bad].any() and (got['b_hop2'][~bad] >= 0).all()


def test_empty_and_one_pair(mods, monkeypatch):
    from oracle import c_oracle
    graph, _ = mods
    n_users, n_biz, eu, eb, pu, pv = corner_graph()
    got = index_and_grouped(monkeypatch, graph, n_users, n_biz, eu, eb, pu[:0], pv[:0])
    assert all(v.size == 0 for v in got.values())
    for i in (0, 15, pu.size - 1):
        got = index_and_grouped(monkeypatch, graph, n_users, n_biz, eu, eb, pu[i:i + 1], pv[i:i + 1])
        check_against(got, c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu[i:i + 1], pv[i:i + 1]), 1)


def test_hop2_is_the_co_review_pattern(mods, monkeypatch):
    """|hop2(b)| as the kernel reports it == row counts of the pattern of A^T A without its diagonal."""
    import scipy.sparse as sp
    graph, synth = mods
    cfg, eu, eb, _, _ = synth.make_config('C1')
    n_users, n_biz = cfg['n_users'], cfg['n_biz']
    A = sp.csr_matrix((np.ones(eu.size, np.int64), (eu, eb)), shape=(n_users, n_biz))
    A.data[:] = 1                                           # duplicates collapse
    C = (A.T @ A).tocsr()
    C.setdiag(0)
    C.eliminate_zeros()
    want = np.diff(C.indptr)
    deg_u = np.bincount(eu, minlength=n_users)
    u0 = int(np.nonzero(deg_u > 0)[0][0])
    pv = np.arange(n_biz, dtype=np.int32)
    pu = np.full(n_biz, u0, np.int32)
    G = handle(monkeypatch, graph, n_users, n_biz, eu, eb)
    got = G.score_pairs_host(pu, pv, want_hop2=True)
    assert biz_path(G) == pkg('_lib').PATH_BIZ_INDEX
    assert np.array_equal(got['b_hop2'].astype(np.int64), want)


def test_selection_and_entry_points(mods, monkeypatch):
    """The override and the cap force the grouped path, a ranged handle reports it, and every entry
    point that reaches the business side gives the same columns."""
    import torch
    graph, synth = mods
    lib = pkg('_lib')
    n_users, n_biz = 20_000, 5000                     # rows: 5000 x 160 words = 3.2 MB
    eu, eb = synth.make_graph(n_users, n_biz, 80_000, seed=21, shift_u=3.0, shift_b=3.0)
    pu, pv = synth.make_pairs(n_users, n_biz, eu, eb, 60_000, k=12, seed=22, invalid_frac=0.01)
    G = handle(monkeypatch, graph, n_users, n_biz, eu, eb)
    info = G.info()
    assert info['biz_index_bytes'] == 5000 * 160 * 4 and info['biz_index_build_ms'] > 0
    capped = handle(monkeypatch, graph, n_users, n_biz, eu, eb, BLP_BIZ_INDEX_MAX_MB=1)
    assert capped.info()['biz_index_bytes'] == 0
    forced = handle(monkeypatch, graph, n_users, n_biz, eu, eb, BLP_BIZ_INDEX_MAX_MB=1, BLP_BIZ_INDEX=1)
    assert forced.info()['biz_index_bytes'] > 0
    ranged = handle(monkeypatch, graph, n_users, n_biz, eu, eb, BLP_RANGES=3)
    assert ranged.info()['biz_index_bytes'] == 0

    du, dv = torch.from_numpy(pu).cuda(), torch.from_numpy(pv).cuda()
    ref = G.score_pairs(du, dv, want_hop2=True, concurrent=False)
    st = G.score_stats(lib.SIDE_BUSINESS)
    assert st['path'] == lib.PATH_BIZ_INDEX and st['range_passes'] == 1
    assert st['group_ms'] == 0 and st['light_ms'] == 0 and st['score_ms'] > 0
    assert st['ctas'] > 0 and st['threads_per_cta'] > 0
    assert G.score_stats(lib.SIDE_USER)['path'] == lib.PATH_GROUPED
    ref = {k: v.cpu().numpy() for k, v in ref.items()}
    runs = {'concurrent': {k: v.cpu().numpy() for k, v in
                           G.score_pairs(du, dv, want_hop2=True, concurrent=True).items()}}
    side = G.score_side(lib.SIDE_BUSINESS, du, dv, want_hop2=True)
    runs['score_side'] = {'b_' + k: v.cpu().numpy() for k, v in side.items()}
    runs['host_session'] = G.host_session(pu.size, columns='all').score(pu, pv)
    for name, H in (('capped', capped), ('forced', forced), ('ranged', ranged)):
        runs[name] = H.score_pairs_host(pu, pv, want_hop2=True)
        want_path = lib.PATH_BIZ_INDEX if name == 'forced' else lib.PATH_GROUPED
        assert biz_path(H) == want_path, name
    assert ranged.score_stats(lib.SIDE_BUSINESS)['range_passes'] >= 2
    for name, got in runs.items():
        for k, v in got.items():
            assert np.array_equal(np.asarray(v), ref[k]), (name, k)
