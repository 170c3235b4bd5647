"""CPU tests of tools/biz_sectors.py: the tests it counts are the kernel's, and the symmetric lookup
it models (row max rank, column min) reads the same bits as row rank(b), column rank(b')."""
import importlib.util
import os

import numpy as np

from conftest import ROOT, pkg


def tool():
    spec = importlib.util.spec_from_file_location('biz_sectors', os.path.join(ROOT, 'tools', 'biz_sectors.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_bitmap_words():
    bs = tool()
    assert bs.bitmap_words(5000) == 160        # the index row of test_gpu_biz_index's 5000 businesses
    assert bs.bitmap_words(61000) == 1908      # C2: 465,552,000 bytes over 61000 rows
    assert all(bs.bitmap_words(n) % 4 == 0 and bs.bitmap_words(n) * 32 > n for n in range(1, 300))


def test_tests_and_symmetric_bits():
    bs = tool()
    synth = pkg('synth')
    n_users, n_biz = 400, 150
    eu, eb = synth.make_graph(n_users, n_biz, 2500, seed=3, shift_u=2.0, shift_b=2.0)
    eu, eb = np.concatenate([eu, eu[:50]]), np.concatenate([eb, eb[:50]])     # duplicate edges
    pu, pv = synth.make_pairs(n_users, n_biz, eu, eb, 3000, k=8, seed=4, invalid_frac=0.01)
    b, bp, rank, n_valid = bs.tests({'n_users': n_users, 'n_biz': n_biz}, eu, eb, pu, pv)

    adj = np.zeros((n_users, n_biz), bool)
    adj[eu, eb] = True
    want_b, want_bp, valid = [], [], 0
    for u, x in zip(pu, pv):                 # one test per b' of N(u) for every pair the kernel scores
        if 0 <= u < n_users and 0 <= x < n_biz and adj[u].any() and adj[:, x].any():
            valid += 1
            want_b += [x] * int(adj[u].sum())
            want_bp += np.nonzero(adj[u])[0].tolist()
    assert n_valid == valid and b.tolist() == want_b and bp.tolist() == want_bp
    # ranks as build_biz_index makes them: de-duplicated degree descending, ties by id
    assert np.array_equal(np.argsort(rank), np.lexsort((np.arange(n_biz), -adj.sum(0))))

    # the index as the device builds it: row rank(b) = hop2(b) over ranks, diagonal clear
    co = (adj.T.astype(int) @ adj.astype(int)) > 0
    np.fill_diagonal(co, False)
    index = np.zeros((n_biz, n_biz), bool)
    index[np.ix_(rank, rank)] = co
    rb, rbp = rank[b], rank[bp]
    direct = index[rb, rbp]
    assert direct.any() and not direct.all()
    assert np.array_equal(index[np.maximum(rb, rbp), np.minimum(rb, rbp)], direct)
    assert np.array_equal(index, index.T)
