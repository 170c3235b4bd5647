"""Every scoring path gives the same answer.

The user/business side of one call is served by up to three mechanisms -- the CTA-per-group kernel
(shared-memory bitmap), the warp-per-group kernel (hash table; hub-free and one-hub groups) and,
inside both, the probe / table path for partners that have a bitmap.  Which one a pair takes
depends on thresholds read at graph creation (BLP_* tuning variables).  These tests force small
graphs through every combination and require (a) bit-identical outputs across the combinations and
(b) agreement with the C oracle.

A handle that fits a business index scores the business side with it, so every combination but
the library defaults also sets BLP_BIZ_INDEX=0: the business side then takes the grouped path (sort
mode, result records and un-permute, the warp-per-group kernel and hub tables), the only one for
graphs too large for an index and for ranged handles, and the defaults compare the index against it.
"""
import numpy as np
import pytest

from conftest import pkg
from test_gpu_parity import check_against, mods  # noqa: F401

pytestmark = pytest.mark.gpu

TUNING = ('BLP_LIGHT', 'BLP_LIGHT_HUBS', 'BLP_PROBE_MIN_DEG', 'BLP_PROBE_RATIO', 'BLP_HUB_MIN_DEG',
          'BLP_BIZ_INDEX')
GROUPED = dict(BLP_BIZ_INDEX='0')   # the business side without the index

# (light kernel, one-hub groups in it, probe bitmaps from this degree on [0 = off], ratio, OR-hub degree)
COMBOS = [
    dict(GROUPED, BLP_LIGHT='0', BLP_PROBE_MIN_DEG='0', BLP_HUB_MIN_DEG='0'),     # CTA kernel, lists only
    dict(GROUPED, BLP_LIGHT='0', BLP_PROBE_MIN_DEG='0', BLP_HUB_MIN_DEG='150'),   # + hub bitmaps
    dict(GROUPED, BLP_LIGHT='0', BLP_PROBE_MIN_DEG='64', BLP_HUB_MIN_DEG='150', BLP_PROBE_RATIO='1'),
    dict(GROUPED, BLP_LIGHT='1', BLP_PROBE_MIN_DEG='0', BLP_HUB_MIN_DEG='150'),   # warp kernel, no probing
    dict(GROUPED, BLP_LIGHT='1', BLP_LIGHT_HUBS='0', BLP_PROBE_MIN_DEG='64', BLP_HUB_MIN_DEG='150'),
    dict(GROUPED, BLP_LIGHT='1', BLP_LIGHT_HUBS='1', BLP_PROBE_MIN_DEG='64', BLP_HUB_MIN_DEG='150',
         BLP_PROBE_RATIO='1'),
    dict(GROUPED, BLP_LIGHT='1', BLP_LIGHT_HUBS='1', BLP_PROBE_MIN_DEG='64', BLP_HUB_MIN_DEG='64',
         BLP_PROBE_RATIO='4'),
    dict(),                                                                  # library defaults
]


def score_with(monkeypatch, graph, env, n_users, n_biz, eu, eb, pu, pv):
    """Scores both sides on a handle created under exactly `env` and checks which path its
    business side took: grouped under BLP_BIZ_INDEX=0, else the index (these graphs are small)."""
    lib = pkg('_lib')
    for k in TUNING:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    G = graph.BipartiteGraph(n_users, n_biz, eu, eb)
    out = G.score_pairs_host(pu, pv, want_hop2=True)
    want_path = lib.PATH_GROUPED if env.get('BLP_BIZ_INDEX') == '0' else lib.PATH_BIZ_INDEX
    assert G.score_stats(lib.SIDE_BUSINESS)['path'] == want_path, env
    info = G.info()
    G.close()
    return out, info


def pairs_with_edges(synth, n_users, n_biz, eu, eb, n_pairs, k, seed):
    """Candidate pairs plus, for every tenth example user, one of the user's OWN businesses
    (a candidate that is already an edge: x is in N(y), which the table path must subtract)."""
    pu, pv = synth.make_pairs(n_users, n_biz, eu, eb, n_pairs, k=k, seed=seed, invalid_frac=0.01)
    first = {}
    for u, b in zip(eu.tolist(), eb.tolist()):
        first.setdefault(u, b)
    pu, pv = pu.copy(), pv.copy()
    for i in range(0, pu.size, 10 * k):
        if pu[i] >= 0:
            pv[i] = first[int(pu[i])]
    return pu, pv


@pytest.mark.parametrize('seed,n_users,n_biz,n_rev,k,alpha_b', [
    (5, 6000, 300, 30000, 16, 2.1),     # a few businesses of several hundred users
    (6, 4000, 120, 24000, 40, 1.9),     # heavier tail, more than 32 pairs per user (two tiles)
    (7, 20000, 2000, 60000, 8, 2.3),    # sparse: most users light, most lists short
])
def test_all_paths_agree(mods, monkeypatch, seed, n_users, n_biz, n_rev, k, alpha_b):
    from oracle import c_oracle
    graph, synth = mods
    eu, eb = synth.make_graph(n_users, n_biz, n_rev, seed=seed, alpha_b=alpha_b, shift_u=3.0,
                              shift_b=2.0)
    pu, pv = pairs_with_edges(synth, n_users, n_biz, eu, eb, 60_000, k, seed + 50)
    want = c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu, pv)
    base, seen = None, set()
    for env in COMBOS:
        got, info = score_with(monkeypatch, graph, env, n_users, n_biz, eu, eb, pu, pv)
        seen.add((info['n_hub_biz'] > 0, env.get('BLP_LIGHT', '1')))
        check_against(got, want, pu.size)
        if base is None:
            base = got
        else:
            for key in base:
                assert np.array_equal(np.asarray(got[key]), np.asarray(base[key])), (env, key)
    # the thresholds really produced hub bitmaps on these shapes (else the test proves nothing)
    assert (True, '1') in seen and (True, '0') in seen


def test_business_side_light_groups_and_unsorted_input(mods, monkeypatch):
    """Pairs in random order (sort-mode grouping, record + un-permute epilogue) through the
    warp-per-group kernel on both sides (the business side without the index)."""
    from oracle import c_oracle
    graph, synth = mods
    n_users, n_biz = 8000, 3000
    eu, eb = synth.make_graph(n_users, n_biz, 40000, seed=9, shift_u=3.0, shift_b=3.0)
    pu, pv = pairs_with_edges(synth, n_users, n_biz, eu, eb, 80_000, 20, 59)
    perm = np.random.default_rng(3).permutation(pu.size)
    pu, pv = pu[perm].copy(), pv[perm].copy()
    want = c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu, pv)
    for env in (dict(GROUPED, BLP_HUB_MIN_DEG='100', BLP_PROBE_MIN_DEG='64'), dict(GROUPED, BLP_LIGHT='0')):
        got, _ = score_with(monkeypatch, graph, env, n_users, n_biz, eu, eb, pu, pv)
        check_against(got, want, pu.size)


def test_light_group_corner_cases(mods, monkeypatch):
    """Hand-made: an isolated star (hop-2 set empty), a user whose only business is a hub, the
    hub itself as the candidate, a candidate that is the user's own business."""
    from oracle import c_oracle
    graph, synth = mods
    n_users, n_biz = 400, 12
    eu, eb = [], []
    for u in range(300):            # business 0 is a hub with 300 users
        eu.append(u); eb.append(0)
    for u in range(0, 300, 3):      # business 1 shares a third of them
        eu.append(u); eb.append(1)
    for u in range(100, 180):       # business 2: 80 users, overlaps both
        eu.append(u); eb.append(2)
    eu += [350]; eb += [5]          # isolated star: user 350 alone at business 5
    eu += [351, 352]; eb += [6, 6]  # two users sharing business 6 only
    eu += [351]; eb += [0]          # ... one of them also in the hub
    eu, eb = np.array(eu, np.int32), np.array(eb, np.int32)
    users = [0, 1, 3, 100, 101, 299, 350, 351, 352, 399]
    pu = np.repeat(np.array(users, np.int32), n_biz)
    pv = np.tile(np.arange(n_biz, dtype=np.int32), len(users))
    want = c_oracle.score_pair_arrays(n_users, n_biz, eu, eb, pu, pv)
    for env in (dict(GROUPED, BLP_HUB_MIN_DEG='200', BLP_PROBE_MIN_DEG='64', BLP_PROBE_RATIO='1'),
                dict(GROUPED, BLP_HUB_MIN_DEG='64', BLP_PROBE_MIN_DEG='64'),
                dict(GROUPED, BLP_LIGHT='0', BLP_HUB_MIN_DEG='200', BLP_PROBE_MIN_DEG='64'),
                dict()):
        got, _ = score_with(monkeypatch, graph, env, n_users, n_biz, eu, eb, pu, pv)
        check_against(got, want, pu.size)


def test_host_buffer_entry_point(mods):
    """blp_score_pairs_host (host buffers in and out, copies inside the call) == the device call,
    for pinned session buffers and for plain pageable numpy arrays.  At 100,000 pairs every plan
    collapses to one user slice and one business slice (slices are at least 65536 pairs); plans
    with several slices are tested in test_gpu_entry_points.test_host_pipeline_slice_plan."""
    import ctypes
    graph, synth = mods
    lib_mod = pkg('_lib')
    cfg, eu, eb, pu, pv = synth.make_config('C1', n_pairs=100_000)
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb)
    want = G.score_pairs_host(pu, pv)            # device call + explicit copies
    n = pu.size
    sess = G.host_session(n, columns='all')
    for plan in ((0, -1, 0), (1, 0, 1), (3, 2, 1), (7, 1, 4)):
        got = sess.score(pu, pv) if plan == (0, -1, 0) else None
        if got is None:
            hu, hb = sess.pinned_inputs(n)
            hu[:] = pu
            hb[:] = pv
            got = sess.score_pinned(n, *plan)
        for k in sess.KEYS:
            assert np.array_equal(got[k], want[k]), (plan, k)
    # pageable memory straight through ctypes
    cols = [np.empty(n, dt) for dt in (np.int32, np.int32, np.float64, np.float64) * 2] + [np.empty(n, np.int64)]
    pu_c, pv_c = np.ascontiguousarray(pu), np.ascontiguousarray(pv)
    rc = G._lib.blp_score_pairs_host(G._h, pu_c.ctypes.data, pv_c.ctypes.data, n,
                                     *[c.ctypes.data for c in cols], 0, -1, 0)
    assert rc == lib_mod.BLP_OK
    for k, c in zip(sess.ALL_KEYS, cols):
        assert np.array_equal(c, want[k]), k
    # a NULL column is skipped (not copied back); no column at all is refused; n = 0 is a no-op
    some = [c.ctypes.data for c in cols]
    cols[3][:] = -7.0
    some[3] = None
    some[5] = None
    cols[0][:] = 0
    assert G._lib.blp_score_pairs_host(G._h, pu_c.ctypes.data, pv_c.ctypes.data, n, *some, 2, 1, 1) \
        == lib_mod.BLP_OK
    assert np.array_equal(cols[0], want['u_cn']) and np.all(cols[3] == -7.0)
    assert G._lib.blp_score_pairs_host(G._h, pu_c.ctypes.data, pv_c.ctypes.data, n, *([None] * 9),
                                       0, -1, 0) == lib_mod.BLP_ERR_INVALID
    assert G._lib.blp_score_pairs_host(G._h, None, None, 0, *([None] * 9), 0, -1, 0) == lib_mod.BLP_OK
