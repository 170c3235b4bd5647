"""Pins the oracles to the reference ITSELF (CPU).

oracle/_ref holds the reference's own similarity.py / util.py as bytecode (oracle/build_ref.py:
three mechanical Python-2 -> 3 rewrites, nothing else), executed by oracle/ref_runner.py with a
stand-in for the stripped SNAP binding.  Two kinds of test:

  * fixture tests   -- tests/golden/cases.json and ref_files.json were WRITTEN by that code
                       (tests/golden/make_golden.py); Oracle A must reproduce them.  These run
                       anywhere, also where /root/reference is absent.
  * live tests      -- run the reference's code here and compare with Oracle A on the fixtures,
                       the known-answer table and hypothesis-generated graphs.  They need
                       oracle/_ref (built from /root/reference in this container; the built files
                       travel to the GPU box) and say so when it is missing.
"""
import json
import os

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

from conftest import pkg
from oracle import build_ref
from oracle import ref_runner as rr
from oracle import similarity_oracle as oa

HERE = os.path.dirname(__file__)
REF_KEYS = ('u_cn', 'u_jaccard', 'u_adamic', 'b_cn', 'b_jaccard', 'b_adamic', 'in_graph')
HAVE_REF = rr.ensure_built()
needs_ref = pytest.mark.skipif(not HAVE_REF, reason='runs the original project\'s own code: oracle/_ref is '
                                                    'not built (oracle/build_ref.py needs a checkout of it)')


def typed_equal(a, b, rtol=0.0):
    """Equal values AND equal Python types (the reference writes int 0 where nothing contributes)."""
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert type(x) is type(y), (x, y)
        if isinstance(x, float) and rtol:
            assert x == pytest.approx(y, rel=rtol, abs=0.0)
        else:
            assert x == y


def test_print_rewrite_rules():
    """The mechanical rewrites of build_ref, on snippets written for this test."""
    src = 'def f(a):\n\tprint "x"\n\tprint "a", a\n\tprint "%d," % a,\n\tprint("kept")\n\tprint "{}".format(a,\n\t\ta),\n'
    out = build_ref.to_python3(src)
    assert 'print("x")' in out and 'print("a", a)' in out
    assert 'print("%d," % a, end=\' \')' in out and 'print("kept")' in out
    assert 'a), end=\' \')' in out
    compile(out, '<t>', 'exec')
    assert build_ref.to_python3('from sets import Set\nx = Set()\n') == 'Set = set\nx = Set()\n'
    # a tab after spaces advances to the next multiple of 8, as Python 2 reads it
    assert build_ref.to_python3('    \tx') == '        x'


def test_fixtures_say_where_they_come_from():
    doc = json.load(open(os.path.join(HERE, 'golden', 'cases.json')))
    assert 'oracle/_ref' in doc['generator'] and set(doc['from_reference']) == set(REF_KEYS)
    assert set(doc['reference_files']) == {'similarity.py', 'util.py'}
    if HAVE_REF:       # the fixtures were made from the reference sources present now
        assert rr.manifest()['files'] == doc['reference_files']


def fixture_shapes(c):
    """The awkward inputs a case puts before the reference (local indices, -1 = invalid id)."""
    eu, eb = np.array(c['edge_u']), np.array(c['edge_b'])
    pu, pv = np.array(c['pair_u']), np.array(c['pair_b'])
    key = eu * c['n_biz'] + eb
    uniq = np.unique(key)
    deg_u = np.bincount(uniq // c['n_biz'], minlength=c['n_users'])
    deg_b = np.bincount(uniq % c['n_biz'], minlength=c['n_biz'])
    ok = (pu >= 0) & (pv >= 0)
    return {'duplicate_edges': key.size > uniq.size,
            'invalid_ids': bool((~ok).any()),
            'isolated_users': bool((deg_u == 0).any()),
            'isolated_businesses': bool((deg_b == 0).any()),
            'degree_one_users': bool((deg_u == 1).any()),
            'degree_one_businesses': bool((deg_b == 1).any()),
            'hub_business': int(deg_b.max()) * 4 >= c['n_users'],     # a quarter of all users
            'pairs_that_are_edges': bool(np.isin(pu[ok] * c['n_biz'] + pv[ok], uniq).any()),
            'pairs_with_isolated_ids': bool((ok & (deg_u[np.clip(pu, 0, None)] == 0)).any()
                                            or (ok & (deg_b[np.clip(pv, 0, None)] == 0)).any())}


def test_oracle_a_reproduces_the_reference_fixtures():
    synth = pkg('synth')
    cases = json.load(open(os.path.join(HERE, 'golden', 'cases.json')))['cases']
    assert len(cases) >= 6
    # what the reference was run on: every awkward shape occurs in some case, so Oracle A is pinned
    # to the reference's own answers on each of them wherever the reference itself is absent
    shapes = [fixture_shapes(c) for c in cases]
    for s in shapes[0]:
        assert any(x[s] for x in shapes), s
    for c in cases:
        ids_eu, ids_eb = synth.shared_ids(c['n_users'], np.array(c['edge_u']), np.array(c['edge_b']))
        ids_pu, ids_pv = synth.shared_ids(c['n_users'], np.array(c['pair_u']), np.array(c['pair_b']))
        got = oa.score_pair_arrays(ids_eu, ids_eb, ids_pu, ids_pv)
        for k in REF_KEYS:
            typed_equal(got[k], c['expect'][k], rtol=1e-15 if 'adamic' in k else 0.0)


def test_oracle_a_files_equal_the_reference_files(tmp_path):
    """File level: Oracle A's main() with the :102 bug reproduced writes what the reference wrote."""
    util = pkg('util')
    doc = json.load(open(os.path.join(HERE, 'golden', 'ref_files.json')))
    (tmp_path / 'graph.txt').write_text(doc['graph_txt'])
    util.write_json(doc['examples'], str(tmp_path / 'examples.json'))
    names = ['u_cn', 'u_jaccard', 'u_adamic', 'b_cn', 'b_jaccard', 'b_adamic']
    paths = [str(tmp_path / (n + '.json')) for n in names]
    M = ['common_neighbors', 'jaccard', 'adamic_adar']
    oa.main(str(tmp_path / 'examples.json'), str(tmp_path / 'graph.txt'), M, paths[:3], M, paths[3:],
            reproduce_reference_bug=True)
    for n, p in zip(names, paths):
        got, want = util.load_json(p), doc['score_files'][n]
        assert got.keys() == want.keys(), n
        for u in want:
            assert got[u].keys() == want[u].keys(), (n, u)
            keys = list(want[u])
            typed_equal([got[u][v] for v in keys], [want[u][v] for v in keys],
                        rtol=1e-15 if 'adamic' in n else 0.0)
    # the reference's b_adamic file: literal zeros of out-of-graph pairs only (similarity.py:102)
    b_ad = doc['score_files']['b_adamic']
    assert all(s == 0 for v in b_ad.values() for s in v.values())
    assert sum(len(v) for v in b_ad.values()) < sum(len(v) for v in doc['examples'].values())


@needs_ref
def test_reference_runs_and_matches_known_answer_table():
    ka = json.load(open(os.path.join(HERE, 'golden', 'known_answer.json')))
    lines = np.array(ka['graph_lines'])
    pu = [p['u'] for p in ka['pairs']]
    pv = [p['v'] for p in ka['pairs']]
    got = rr.score_pair_arrays(lines[:, 0], lines[:, 1], pu, pv)
    for k in ('u_cn', 'u_jaccard', 'u_adamic', 'b_cn', 'b_jaccard', 'b_adamic'):
        # the hand-checked table carries the reference's types (int 0 vs 0.0) as well
        typed_equal(got[k], [p[k] for p in ka['pairs']], rtol=1e-15 if 'adamic' in k else 0.0)
    assert got['in_graph'] == [1] * 8 + [0, 0]
    assert got['b_adamic_file'] == [None] * 8 + [0, 0]      # the dead branch, as the reference has it


@needs_ref
def test_reference_reproduces_its_own_fixtures():
    """Guards against stale fixtures: the code in oracle/_ref still writes what cases.json holds."""
    synth = pkg('synth')
    cases = json.load(open(os.path.join(HERE, 'golden', 'cases.json')))['cases']
    for c in cases[:4]:
        ids_eu, ids_eb = synth.shared_ids(c['n_users'], np.array(c['edge_u']), np.array(c['edge_b']))
        ids_pu, ids_pv = synth.shared_ids(c['n_users'], np.array(c['pair_u']), np.array(c['pair_b']))
        got = rr.score_pair_arrays(ids_eu, ids_eb, ids_pu, ids_pv)
        for k in REF_KEYS:
            typed_equal(got[k], c['expect'][k], rtol=1e-15 if 'adamic' in k else 0.0)


graphs = st.tuples(st.integers(2, 25), st.integers(2, 12), st.integers(0, 2 ** 31 - 1),
                   st.integers(1, 120))


@needs_ref
@settings(max_examples=30, deadline=None, suppress_health_check=list(HealthCheck))
@given(graphs)
def test_oracle_a_equals_the_reference_on_random_graphs(g):
    n_users, n_biz, seed, n_edges = g
    rng = np.random.default_rng(seed)
    eu = rng.integers(0, n_users, n_edges)          # duplicates, isolated ids, degree-1 nodes, hubs
    eb = rng.integers(0, n_biz, n_edges) if seed % 3 else np.minimum(rng.geometric(0.5, n_edges) - 1, n_biz - 1)
    pu = rng.integers(-1, n_users, 60)
    pv = rng.integers(-1, n_biz, 60)
    synth = pkg('synth')
    ids_eu, ids_eb = synth.shared_ids(n_users, eu, eb)
    ids_pu, ids_pv = synth.shared_ids(n_users, pu, pv)
    ref = rr.score_pair_arrays(ids_eu, ids_eb, ids_pu, ids_pv)
    port = oa.score_pair_arrays(ids_eu, ids_eb, ids_pu, ids_pv)
    for k in REF_KEYS:
        # same sets, but the reference sums adamic_adar in ITS set-iteration order
        typed_equal(ref[k], port[k], rtol=1e-12 if 'adamic' in k else 0.0)
