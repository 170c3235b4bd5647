"""The entry points and arguments that a default call never reaches, on one GPU.

* blp_score_pairs_host with more than one slice.  Slices are at least 65536 pairs, so the
  workload has 600,003 pairs (up to 9 slices, odd, most bounds off a multiple of four): lead
  upload, business slices between user slices, copy-back of later slices, NULL columns, staging
  buffers that grow between calls.
* blp_derive_pairs, blp_peer_push and the dist.ResultWindow layout within one process: derived
  jaccard and pa must be bit-identical to what the kernels write.
* blp_score_pairs with one output at a time, ids and outputs at odd element offsets, and canaries
  behind every output (a call writes n elements, no more), on every epilogue: user side grouped by
  runs and by sort, business index, grouped business side (records + un-permute), ranged handle.
* Adamic-Adar is exact: the weights are llrint(2^31 / ln d) and every path adds them as integers,
  so the output is (sum of the Q1.31 weights) / 2^31 bit for bit.  exact_adamic restates that with
  scipy in int64; every test here that gets adamic back holds it to that value.
* blp_graph_reserve_sms.

The reference of each comparison is the plain device call (score_pairs), itself held to the exact
Adamic-Adar value and, on one combination, to the C oracle.
"""
import ctypes
import math

import numpy as np
import pytest

from conftest import pkg
from test_gpu_parity import check_against, mods  # noqa: F401
from test_gpu_paths import COMBOS, GROUPED, TUNING, pairs_with_edges, score_with

pytestmark = pytest.mark.gpu

N = 600_003
ORDERS = ('grouped', 'permuted')
# blp_score_pairs_host's output arguments, in order
HOST_KEYS = ('u_cn', 'u_union', 'u_jaccard', 'u_adamic', 'b_cn', 'b_union', 'b_jaccard', 'b_adamic', 'pa')
KINDS = ('cn', 'union', 'jaccard', 'adamic', 'pa', 'hop2')
NP_DTYPE = {'cn': np.int32, 'union': np.int32, 'jaccard': np.float64, 'adamic': np.float64,
            'pa': np.int64, 'hop2': np.int32}
SENTINEL = {'cn': -123456789, 'union': -123456789, 'jaccard': -0.75, 'adamic': -0.75,
            'pa': -(3 << 60), 'hop2': -123456789}     # no output ever takes these values
HOST_TAIL = 16
DEVICE_TAIL = 64
# (user slices, lead slices, business slices); <= 0 / < 0 / <= 0 select the defaults 4 / 1 / 2
PLANS = ((0, -1, 0), (1, 0, 1), (2, 0, 2), (2, 1, 1), (4, 3, 2), (3, 0, 9), (9, 4, 3),
         (50, 100, 50), (3, -5, 0))
ENV = TUNING + ('BLP_RANGES', 'BLP_BIZ_INDEX_MAX_MB')


def kind(col):
    return col if col == 'pa' else col.split('_', 1)[1]


def exact_adamic(n_users, n_biz, edge_u, edge_b, pair_u, pair_b):
    """Q1.31 Adamic-Adar sums of both sides, int64 throughout: (q_user, q_business) per pair.

    User side: sum over users i in hop2(u) & N(b) of w(deg i); hop2(u) is the pattern of A A^T
    without its diagonal, so the sums are M = (H diag(w_user)) A at (u, b).  Business side: the same
    with A^T.  w(d) = round(2^31 / ln d) for d > 1, else 0, with math.log (the host libm, as the
    library's weight table)."""
    import scipy.sparse as sp
    A = sp.csr_matrix((np.ones(len(edge_u), np.int64), (edge_u, edge_b)), shape=(n_users, n_biz))
    A.data[:] = 1                                      # duplicate edges collapse
    At = A.T.tocsr()
    du, db = np.diff(A.indptr), np.diff(At.indptr)

    def weights(deg):
        w = np.zeros(deg.size, np.int64)
        for d in np.unique(deg):
            if d > 1:
                w[deg == d] = round(math.ldexp(1.0 / math.log(int(d)), 31))
        return w
    pu, pv = np.asarray(pair_u, np.int64), np.asarray(pair_b, np.int64)
    ok = (pu >= 0) & (pu < n_users) & (pv >= 0) & (pv < n_biz)
    ok[ok] = (du[pu[ok]] > 0) & (db[pv[ok]] > 0)
    res = []
    for X, Xt, w, px, py in ((A, At, weights(du), pu, pv), (At, A, weights(db), pv, pu)):
        H = (X @ Xt).tocsr()
        H.setdiag(0)
        H.eliminate_zeros()
        H.data[:] = w[H.indices]                       # H diag(w), pattern only
        M = (H @ X).tocsr()
        assert M.dtype == np.int64
        q = np.zeros(pu.size, np.int64)
        q[ok] = np.asarray(M[px[ok], py[ok]]).ravel()
        res.append(q)
    return res[0], res[1]


def first_diff(a, b):
    bad = np.nonzero(a != b)[0]
    return '%d rows differ, first %s: got %s want %s' % (bad.size, bad[:4], a[bad[:4]], b[bad[:4]])


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def assert_exact_adamic(got, qu, qb, what=''):
    """got['u_adamic'] / got['b_adamic'] (those present) == q / 2^31 bit for bit."""
    checked = 0
    for col, q in (('u_adamic', qu), ('b_adamic', qb)):
        if col in got:
            g = np.asarray(got[col])[:q.size]
            want = q / 2.0 ** 31
            assert same_bits(g, want), (what, col, first_diff(g, want))
            checked += 1
    return checked


def assert_host_columns(got, want, n, qu, qb, what=''):
    """Host columns of n + HOST_TAIL rows: the first n bit-identical to `want`, the tail untouched,
    adamic exact."""
    for k, v in got.items():
        assert same_bits(v[:n], want[k][:n]), (what, k, first_diff(v[:n], want[k][:n]))
        assert np.all(v[n:] == SENTINEL[kind(k)]), (what, k, 'written past n')
    assert_exact_adamic({k: v[:n] for k, v in got.items()}, qu[:n], qb[:n], what)


def host_columns(n, keys=HOST_KEYS):
    return {k: np.full(n + HOST_TAIL, SENTINEL[kind(k)], NP_DTYPE[kind(k)]) for k in keys}


def host_call(G, pu, pv, cols, plan):
    """blp_score_pairs_host on pageable numpy arrays; columns not in `cols` are NULL."""
    ptrs = [cols[k].ctypes.data if k in cols else None for k in HOST_KEYS]
    return G._lib.blp_score_pairs_host(G._h, pu.ctypes.data, pv.ctypes.data, int(pu.size), *ptrs, *plan)


def make_handle(graph, w, **env):
    """A C1 handle created under exactly `env` (the tuning variables are read at creation)."""
    with pytest.MonkeyPatch.context() as mp:
        for k in ENV:
            mp.delenv(k, raising=False)
        for k, v in env.items():
            mp.setenv(k, str(v))
        return graph.BipartiteGraph(w['n_users'], w['n_biz'], w['eu'], w['eb'])


@pytest.fixture(scope='module')
def c1(mods):
    """C1's graph with N pairs, grouped by user and permuted, with the exact adamic of each."""
    graph, synth = mods
    cfg, eu, eb, pu, pv = synth.make_config('C1', n_pairs=N)
    assert pu.size == N
    qu, qb = exact_adamic(cfg['n_users'], cfg['n_biz'], eu, eb, pu, pv)
    perm = np.random.default_rng(17).permutation(N)
    orders = {'grouped': (pu, pv, qu, qb), 'permuted': (pu[perm], pv[perm], qu[perm], qb[perm])}
    # another list of the same length: scored in between so that rows a call leaves unwritten show
    # other numbers than the ones expected
    decoy = (np.ascontiguousarray(pu[::-1]), np.ascontiguousarray(pv[::-1]))
    return dict(n_users=cfg['n_users'], n_biz=cfg['n_biz'], eu=eu, eb=eb, orders=orders, perm=perm,
                decoy=decoy)


@pytest.fixture(scope='module')
def handles(mods, c1):
    """'index': the default handle (business index); 'grouped': BLP_BIZ_INDEX=0 (the business side
    groups by sort, writes records and un-permutes them)."""
    graph, _ = mods
    hs = {'index': make_handle(graph, c1), 'grouped': make_handle(graph, c1, BLP_BIZ_INDEX=0)}
    assert hs['index'].info()['biz_index_bytes'] > 0 and hs['grouped'].info()['biz_index_bytes'] == 0
    yield hs
    for G in hs.values():
        G.close()


@pytest.fixture(scope='module')
def ref(handles, c1):
    """The plain device call (score_pairs) per (handle, order), hop2 included, on the host."""
    import torch
    lib = pkg('_lib')
    out = {}
    for name, G in handles.items():
        for order in ORDERS:
            pu, pv, _, _ = c1['orders'][order]
            r = G.score_pairs(torch.from_numpy(pu).to(G.device), torch.from_numpy(pv).to(G.device),
                              want_hop2=True)
            torch.cuda.synchronize(G.device)
            want_path = lib.PATH_BIZ_INDEX if name == 'index' else lib.PATH_GROUPED
            assert G.score_stats(lib.SIDE_BUSINESS)['path'] == want_path
            out[name, order] = {k: v.cpu().numpy() for k, v in r.items()}
    return out


@pytest.fixture(scope='module')
def sessions(handles):
    return {name: G.host_session(N + HOST_TAIL, columns='all') for name, G in handles.items()}


# ------------------------------------------------------------------------------------ reference
def test_reference_is_exact_and_matches_the_oracle(c1, ref):
    from oracle import c_oracle
    for (name, order), got in ref.items():
        _, _, qu, qb = c1['orders'][order]
        assert assert_exact_adamic(got, qu, qb, (name, order)) == 2
        other = ref['index', order]
        for k in got:
            assert same_bits(got[k], other[k]), (name, order, k)
    # the permuted order holds the same rows
    for k, v in ref['grouped', 'grouped'].items():
        assert same_bits(v[c1['perm']], ref['grouped', 'permuted'][k]), k
    pu, pv = c1['orders']['grouped'][:2]
    want = c_oracle.score_pair_arrays_parallel(c1['n_users'], c1['n_biz'], c1['eu'], c1['eb'], pu, pv)
    check_against(ref['index', 'grouped'], want, N)


# ------------------------------------------------------------------- blp_score_pairs_host
@pytest.mark.parametrize('plan', PLANS, ids=lambda p: '%d/%d/%d' % p)
def test_host_pipeline_slice_plan(c1, handles, ref, sessions, plan):
    """Every slice plan through the pinned session and through pageable numpy: all nine columns
    bit-identical to the device call, nothing written behind row n."""
    du, dv = c1['decoy']
    spare = np.empty(N, np.int64)
    for name, G in handles.items():
        sess = sessions[name]
        for order in ORDERS:
            pu, pv, qu, qb = c1['orders'][order]
            want = ref[name, order]
            what = (plan, name, order)
            # pinned
            assert host_call(G, du, dv, {'pa': spare}, (1, 0, 1)) == 0
            hu, hb = sess.pinned_inputs(N)
            hu[:] = pu
            hb[:] = pv
            for k in sess.KEYS:
                sess.h_out[k].fill_(SENTINEL[kind(k)])
            sess.score_pinned(N, *plan)
            assert_host_columns({k: sess.h_out[k].numpy() for k in sess.KEYS}, want, N, qu, qb,
                                what + ('pinned',))
            # pageable
            assert host_call(G, du, dv, {'pa': spare}, (1, 0, 1)) == 0
            cols = host_columns(N)
            assert host_call(G, pu, pv, cols, plan) == 0
            assert_host_columns(cols, want, N, qu, qb, what + ('pageable',))


@pytest.mark.parametrize('plan', [(9, 4, 3), (4, 1, 2)], ids=lambda p: '%d/%d/%d' % p)
def test_host_pipeline_null_columns(c1, handles, ref, plan):
    """A multi-slice plan asked for a few columns: those are right, nothing else is touched."""
    du, dv = c1['decoy']
    spare = np.empty(N, np.int64)
    for name, G in handles.items():
        for order in ORDERS:
            pu, pv, qu, qb = c1['orders'][order]
            for subset in (('pa',), ('b_adamic',), ('u_cn', 'b_union')):
                assert host_call(G, du, dv, {'pa': spare}, (1, 0, 1)) == 0
                cols = host_columns(N)
                assert host_call(G, pu, pv, {k: cols[k] for k in subset}, plan) == 0
                assert_host_columns({k: cols[k] for k in subset}, ref[name, order], N, qu, qb,
                                    (plan, name, order, subset))
                for k in HOST_KEYS:
                    if k not in subset:
                        assert np.all(cols[k] == SENTINEL[kind(k)]), (name, order, subset, k)


def test_host_pipeline_staging_grows_and_is_reused(mods, c1, ref):
    """One fresh handle: 200k pairs, then N (the staging buffers grow), then 777 (they are reused)."""
    graph, _ = mods
    G = make_handle(graph, c1)
    try:
        for order, n in (('permuted', 200_000), ('grouped', N), ('permuted', 777)):
            pu, pv, qu, qb = c1['orders'][order]
            for plan in ((0, -1, 0), (9, 4, 3)):
                cols = host_columns(n)
                assert host_call(G, pu[:n], pv[:n], cols, plan) == 0
                assert_host_columns(cols, ref['index', order], n, qu[:n], qb[:n], (order, n, plan))
    finally:
        G.close()


# ------------------------------------------------------------------------ blp_derive_pairs
def test_derive_pairs_equals_the_kernels(c1, handles):
    """u_jaccard, b_jaccard and pa from blp_derive_pairs == what the scoring kernels write, on pairs
    with negative, out-of-range and degree-0 ids; over the whole list, over a range that starts at
    an odd offset, one output at a time; argument errors."""
    import torch
    lib = pkg('_lib')
    G = handles['index']
    du, db = G.degrees(lib.SIDE_USER), G.degrees(lib.SIDE_BUSINESS)
    nu, nb = c1['n_users'], c1['n_biz']
    u0, b0 = np.nonzero(du == 0)[0], np.nonzero(db == 0)[0]
    assert u0.size and b0.size
    pu, pv = c1['orders']['permuted'][:2]
    bad_u = [-1, -7, nu, nu + 5, int(u0[0]), int(u0[-1]), 3, 3, int(u0[1])]
    bad_v = [2, 2, 2, -1, 1, 7, nb, int(b0[0]), int(b0[0])]
    pu = np.concatenate([pu[:150_000], np.array(bad_u, np.int32), pu[150_000:200_000]])
    pv = np.concatenate([pv[:150_000], np.array(bad_v, np.int32), pv[150_000:200_000]])
    n = pu.size
    qu, qb = exact_adamic(nu, nb, c1['eu'], c1['eb'], pu, pv)
    d_u, d_b = torch.from_numpy(pu).cuda(G.device), torch.from_numpy(pv).cuda(G.device)
    r = G.score_pairs(d_u, d_b)
    torch.cuda.synchronize(G.device)
    assert_exact_adamic({k: v.cpu().numpy() for k, v in r.items()}, qu, qb)
    st = torch.cuda.current_stream(G.device)

    def at(t, lo):
        return ctypes.c_void_p(t.data_ptr() + t.element_size() * lo) if t is not None else None

    def derive(lo, hi, which):
        m = hi - lo
        out = {k: torch.full((m + DEVICE_TAIL,), SENTINEL[kind(k)], dtype=r[k].dtype, device=G.device)
               for k in which}
        uj, bj, pa = 'u_jaccard' in which, 'b_jaccard' in which, 'pa' in which
        rc = G._lib.blp_derive_pairs(
            G._h, at(d_u if pa else None, lo), at(d_b if pa else None, lo), m,
            at(r['u_cn'] if uj else None, lo), at(r['u_union'] if uj else None, lo),
            at(r['b_cn'] if bj else None, lo), at(r['b_union'] if bj else None, lo),
            at(out.get('u_jaccard'), 0), at(out.get('b_jaccard'), 0), at(out.get('pa'), 0),
            ctypes.c_void_p(st.cuda_stream))
        assert rc == lib.BLP_OK, G._lib.blp_last_error()
        torch.cuda.synchronize(G.device)
        for k, t in out.items():
            got = t.cpu().numpy()
            want = r[k][lo:hi].cpu().numpy()
            assert same_bits(got[:m], want), (lo, hi, which, k, first_diff(got[:m], want))
            assert np.all(got[m:] == SENTINEL[kind(k)]), (lo, hi, which, k, 'written past n')
    derived = ('u_jaccard', 'b_jaccard', 'pa')
    derive(0, n, derived)
    derive(150_001, n - 2, derived)         # odd offset, the invalid ids inside
    for k in derived:
        derive(0, n, (k,))
        derive(149_999, 150_011, (k,))
    # the invalid pairs really are "not in graph" rows
    pa = r['pa'].cpu().numpy()[150_000:150_000 + len(bad_u)]
    assert not pa.any()
    # argument errors
    f = G._lib.blp_derive_pairs
    p = ctypes.c_void_p
    o = torch.empty(n, dtype=torch.float64, device=G.device)
    s = p(st.cuda_stream)
    ptr = lambda t: p(t.data_ptr())   # noqa: E731
    assert f(G._h, None, None, n, None, ptr(r['u_union']), None, None, ptr(o), None, None, s) == lib.BLP_ERR_INVALID
    assert f(G._h, None, None, n, ptr(r['u_cn']), None, None, None, ptr(o), None, None, s) == lib.BLP_ERR_INVALID
    assert f(G._h, None, None, n, None, None, ptr(r['b_cn']), None, None, ptr(o), None, s) == lib.BLP_ERR_INVALID
    assert f(G._h, ptr(d_u), None, n, None, None, None, None, None, None, ptr(r['pa']), s) == lib.BLP_ERR_INVALID
    assert f(G._h, None, ptr(d_b), n, None, None, None, None, None, None, ptr(r['pa']), s) == lib.BLP_ERR_INVALID
    assert f(G._h, None, None, 0, *([None] * 7), s) == lib.BLP_OK
    assert f(G._h, None, None, -1, *([None] * 7), s) == lib.BLP_ERR_INVALID


# ------------------------------------------------------------------- result window, world 1
WINDOWS = {   # columns, derived, bytes per pair on the wire
    'default': ('REFERENCE_COLUMNS', None, 40),
    'all_columns_32': ('ALL_COLUMNS', 'DERIVED_COLUMNS', 32),
    'reference_columns_32': ('REFERENCE_COLUMNS', 'DERIVED_COLUMNS', 32),   # unions kept internally
}


@pytest.mark.parametrize('layout', sorted(WINDOWS))
def test_result_window_world_one(c1, handles, ref, layout):
    """The window on its owner, one process: own rows [lo, hi) by score_into_window, every other
    row the way a peer writes it (the wire columns only: the user side's kernels store into the
    window, the business side goes through local staging and blp_peer_push), then derive().  The
    window must hold what the unsharded call returns."""
    import torch
    lib = pkg('_lib')
    d = pkg('dist')
    G = handles['index']
    pu, pv, qu, qb = c1['orders']['grouped']
    d_u, d_b = torch.from_numpy(pu).cuda(G.device), torch.from_numpy(pv).cuda(G.device)
    cols, which, per_pair = WINDOWS[layout]
    columns = getattr(d, cols)
    which = None if which is None else getattr(d, which)
    window = d.ResultWindow(G, N, columns=columns) if which is None else \
        d.ResultWindow(G, N, columns=columns, derived=which)
    try:
        assert window.world == 1 and window.bytes_per_pair() == per_pair
        wire = d.window_layout(N, columns, True, which)['wire']
        for c, t in window.tensors().items():
            t.fill_(SENTINEL[kind(c)])
        lo, hi = 100_001, 350_003
        st = torch.cuda.current_stream(G.device)
        d.score_into_window(G, d_u[lo:hi], d_b[lo:hi], window, lo)
        u_wire = [c for c in wire if not c.startswith('b_')]
        b_wire = [c for c in wire if c.startswith('b_')]
        for a, b in ((0, lo), (hi, N)):
            p = window.pointers(a, u_wire)
            G.score_side(lib.SIDE_USER, d_u[a:b], d_b[a:b], want=(), out_ptr={kind(c): p[c] for c in u_wire})
            stage = G.score_side(lib.SIDE_BUSINESS, d_u[a:b], d_b[a:b], want=tuple(kind(c) for c in b_wire))
            p = window.pointers(a, b_wire)
            for c in b_wire:
                t = stage[kind(c)]
                lib.check(G._lib.blp_peer_push(G.device.index or 0, ctypes.c_void_p(p[c]),
                                               ctypes.c_void_p(t.data_ptr()), t.numel() * t.element_size(),
                                               ctypes.c_void_p(st.cuda_stream)), 'blp_peer_push')
        window.derive(d_u, d_b, (lo, hi))
        torch.cuda.synchronize(G.device)
        got = {k: v.cpu().numpy() for k, v in window.tensors().items()}
        assert set(got) == set(columns)
        for k, v in got.items():
            assert same_bits(v, ref['index', 'grouped'][k]), (layout, k, first_diff(v, ref['index', 'grouped'][k]))
        assert assert_exact_adamic(got, qu, qb) == 2
    finally:
        torch.cuda.synchronize(G.device)
        window.close()


# ----------------------------------------------- blp_score_pairs: one output at a time, offsets
PATHS = {   # handle, side, pair order
    'user_runs': ('index', 0, 'grouped'),
    'user_sort': ('index', 0, 'permuted'),
    'biz_index': ('index', 1, 'permuted'),
    'biz_grouped': ('grouped', 1, 'permuted'),
    'ranged_user': ('ranged', 0, 'grouped'),
    'ranged_biz': ('ranged', 1, 'permuted'),
}


@pytest.fixture(scope='module')
def ranged(mods, c1):
    graph, _ = mods
    G = make_handle(graph, c1, BLP_RANGES=3)
    assert G.info()['biz_index_bytes'] == 0
    yield G
    G.close()


@pytest.mark.parametrize('path', sorted(PATHS))
def test_score_pairs_one_output_at_a_time(c1, handles, ranged, ref, path):
    """blp_score_pairs with every output, then with each one alone: each equals the full call, the
    full call equals the reference, and nothing is written behind row n.  Then again with the pair
    ids and every output starting one element into their storage."""
    import torch
    lib = pkg('_lib')
    name, side, order = PATHS[path]
    G = ranged if name == 'ranged' else handles[name]
    pu, pv, qu, qb = c1['orders'][order]
    want = ref['index', order]
    s = 'u_' if side == lib.SIDE_USER else 'b_'
    h_u, h_b = torch.from_numpy(pu).cuda(G.device), torch.from_numpy(pv).cuda(G.device)
    for shift in (0, 1):
        d_u, d_b = h_u[shift:], h_b[shift:]
        n = N - shift
        assert d_u.data_ptr() % 8 == 4 * shift

        def outputs():
            return {k: torch.full((shift + n + DEVICE_TAIL,), SENTINEL[k], dtype=getattr(torch, np.dtype(NP_DTYPE[k]).name),
                                  device=G.device)[shift:] for k in KINDS}

        def call(outs, keys):
            G.score_side(side, d_u, d_b, want=(), out_ptr={k: outs[k].data_ptr() for k in keys})
            return outs
        full = call(outputs(), KINDS)
        torch.cuda.synchronize(G.device)
        if name == 'ranged':
            assert G.score_stats(side)['range_passes'] >= 2
        want_path = lib.PATH_BIZ_INDEX if (name == 'index' and side == lib.SIDE_BUSINESS) else lib.PATH_GROUPED
        assert G.score_stats(side)['path'] == want_path
        host = {k: v.cpu().numpy() for k, v in full.items()}
        for k in KINDS:
            col = 'pa' if k == 'pa' else s + k
            assert same_bits(host[k][:n], want[col][shift:]), (path, shift, k, first_diff(host[k][:n], want[col][shift:]))
            assert np.all(host[k][n:] == SENTINEL[k]), (path, shift, k, 'written past n')
        assert assert_exact_adamic({s + 'adamic': host['adamic'][:n]}, qu[shift:], qb[shift:], (path, shift)) == 1
        for k in KINDS:
            one = call(outputs(), (k,))
            torch.cuda.synchronize(G.device)
            assert torch.equal(one[k], full[k]), (path, shift, k)
            for other in KINDS:
                if other != k:
                    assert bool((one[other] == SENTINEL[other]).all()), (path, shift, k, other)


# --------------------------------------------------------------------- exact adamic, every path
def test_adamic_exact_on_every_path(mods, monkeypatch):
    """The graph of test_gpu_paths with the most hub rows, under every combination of its
    thresholds (probe, hub table, warp-per-group kernel, business index) and on a ranged handle."""
    graph, synth = mods
    seed, n_users, n_biz, n_rev, k, alpha_b = 6, 4000, 120, 24000, 40, 1.9
    eu, eb = synth.make_graph(n_users, n_biz, n_rev, seed=seed, alpha_b=alpha_b, shift_u=3.0, shift_b=2.0)
    pu, pv = pairs_with_edges(synth, n_users, n_biz, eu, eb, 60_000, k, seed + 50)
    qu, qb = exact_adamic(n_users, n_biz, eu, eb, pu, pv)
    hubs = 0
    for env in COMBOS + [dict(GROUPED, BLP_RANGES='3')]:   # (score_with leaves BLP_RANGES set: last)
        got, info = score_with(monkeypatch, graph, env, n_users, n_biz, eu, eb, pu, pv)
        assert assert_exact_adamic(got, qu, qb, env) == 2
        hubs += info['n_hub_biz'] > 0 and info['n_hub_users'] > 0
    assert hubs >= 2


# ------------------------------------------------------------------------------ reserve_sms
def test_reserve_sms(c1, handles, ref):
    """Reserving SMs shrinks the persistent grids by exactly that share and changes no result;
    -1 and sm_count are refused."""
    import torch
    lib = pkg('_lib')
    G = handles['grouped']
    sm = G.info()['sm_count']
    pu, pv, qu, qb = c1['orders']['grouped']
    d_u, d_b = torch.from_numpy(pu).cuda(G.device), torch.from_numpy(pv).cuda(G.device)

    def run():
        r = G.score_pairs(d_u, d_b, concurrent=False)
        torch.cuda.synchronize(G.device)
        ctas = [G.score_stats(sd)['ctas'] for sd in (lib.SIDE_USER, lib.SIDE_BUSINESS)]
        return {k: v.cpu().numpy() for k, v in r.items()}, ctas
    base, ctas0 = run()
    assert all(c > 0 and c % sm == 0 for c in ctas0), ctas0
    try:
        for r in (1, sm - 1):
            G.reserve_sms(r)
            got, ctas = run()
            for c, c0 in zip(ctas, ctas0):
                assert c * sm == c0 * (sm - r), (r, ctas, ctas0)
            for k, v in got.items():
                assert same_bits(v, ref['grouped', 'grouped'][k]), (r, k)
            assert assert_exact_adamic(got, qu, qb, r) == 2
        for bad in (-1, sm):
            with pytest.raises(ValueError):
                G.reserve_sms(bad)
    finally:
        G.reserve_sms(0)
    got, ctas = run()
    assert ctas == ctas0
