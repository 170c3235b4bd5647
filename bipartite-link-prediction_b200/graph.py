"""Graph handle: the object that stands where the reference passes a SNAP ``PUNGraph``.

The reference loads ``graph.txt`` with ``snap.LoadEdgeList(snap.PUNGraph, f, 0, 1)``
(similarity.py:16) and then only ever asks the graph for its node ids (:22,:65), BFS hops
(:29,:41,:74,:85) and degrees (:121).  ``BipartiteGraph`` owns the device-resident CSR pair behind
the C ABI (include/blp.h) and offers those SNAP spellings for the set-level helpers; the bulk
scoring goes through ``score_pairs`` -> ``blp_score_pairs`` (CUDA, no CPU path).

PyTorch is used here for device buffers and streams only.
"""
import ctypes
import time

import numpy as np
import torch

from . import _lib

OUTPUTS_PER_SIDE = ('cn', 'union', 'jaccard', 'adamic')


def read_edge_list(path):
    """graph.txt -> two int64 arrays (column 0 = user id, column 1 = business id).

    Format: one ``"<user_id> <business_id>\\n"`` per review, duplicates allowed
    (dataset_maker.py:197).
    """
    try:
        import pandas as pd
        df = pd.read_csv(path, sep=r'\s+', header=None, usecols=[0, 1], dtype=np.int64,
                         engine='c')
        return df[0].to_numpy(), df[1].to_numpy()
    except ImportError:  # pragma: no cover
        arr = np.loadtxt(path, dtype=np.int64, usecols=(0, 1), ndmin=2)
        return arr[:, 0].copy(), arr[:, 1].copy()


def read_edge_list_device(path, device=None):
    """graph.txt -> two int64 CUDA tensors, parsed ON the device (``blp_edge_list_count`` /
    ``blp_edge_list_parse``): the file's bytes are uploaded as they are; data lines are lines
    whose first non-blank character starts an integer (blank / comment lines skipped, columns
    beyond the second ignored).  Raises ValueError when a data line lacks a second integer."""
    lib = _lib.load()
    if device is None:
        device = torch.cuda.current_device()
    dev = device if isinstance(device, torch.device) else torch.device('cuda', int(device))
    raw = np.fromfile(path, dtype=np.uint8)
    with torch.cuda.device(dev):
        text = torch.from_numpy(raw).to(dev)
        st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        n_lines = ctypes.c_int64(0)
        _lib.check(lib.blp_edge_list_count(ctypes.c_void_p(text.data_ptr()), int(text.numel()),
                                           ctypes.byref(n_lines), st), 'blp_edge_list_count')
        n = int(n_lines.value)
        col0 = torch.empty(n, dtype=torch.int64, device=dev)
        col1 = torch.empty(n, dtype=torch.int64, device=dev)
        _lib.check(lib.blp_edge_list_parse(ctypes.c_void_p(text.data_ptr()), int(text.numel()), n,
                                           ctypes.c_void_p(col0.data_ptr()),
                                           ctypes.c_void_p(col1.data_ptr()), st), 'blp_edge_list_parse')
    return col0, col1


class _NodeIt(object):
    """``G.GetNI(i)`` -- only ``GetDeg`` / ``GetId`` are used by the reference (similarity.py:22,121)."""

    def __init__(self, nid, deg):
        self._nid, self._deg = nid, deg

    def GetDeg(self):
        return self._deg

    def GetId(self):
        return self._nid


class BipartiteGraph(object):
    """De-duplicated user x business graph, resident in HBM on one device.

    Two ways in:
      * ``BipartiteGraph(n_users, n_biz, edge_u, edge_b)`` -- LOCAL indices (users 0..n_users-1,
        businesses 0..n_biz-1); nodes that appear on no edge have degree 0 = "not in graph".
      * ``BipartiteGraph.from_id_edges(ids_u, ids_b)`` / ``from_edge_list(path)`` -- the
        reference's shared id space; ids are compacted, and the two columns must be disjoint
        (dataset_maker.py:173-174 guarantees it; hop-2 means something else otherwise).
    """

    def __init__(self, n_users, n_biz, edge_u, edge_b, device=None, user_ids=None, biz_ids=None,
                 build='device'):
        """build='device' (default): blp_graph_create_device -- CUDA int32 tensors are taken as they
        are, anything else is uploaded first; radix sort and CSR build run on the GPU;
        build='host': host int32 arrays are handed to blp_graph_create, which uploads them and runs
        the same build.  Both yield the same graph."""
        lib = _lib.load()
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        if isinstance(device, torch.device):
            device = device.index or 0
        self._lib = lib
        self._h = ctypes.c_void_p()
        if build == 'device':
            dev = torch.device('cuda', int(device))
            with torch.cuda.device(dev):
                def to_dev(x):
                    if isinstance(x, torch.Tensor):
                        return x.to(device=dev, dtype=torch.int32).contiguous()
                    return torch.from_numpy(np.ascontiguousarray(np.asarray(x), dtype=np.int32)).to(dev)
                teu, teb = to_dev(edge_u), to_dev(edge_b)
                if teu.shape != teb.shape or teu.dim() != 1:
                    raise ValueError('edge_u and edge_b must be 1-D arrays of equal length')
                st = torch.cuda.current_stream(dev)
                rc = lib.blp_graph_create_device(int(n_users), int(n_biz), int(teu.numel()),
                                                 ctypes.c_void_p(teu.data_ptr()),
                                                 ctypes.c_void_p(teb.data_ptr()), int(device),
                                                 ctypes.c_void_p(st.cuda_stream),
                                                 ctypes.byref(self._h))
            _lib.check(rc, 'blp_graph_create_device')
        elif build == 'host':
            eu = np.ascontiguousarray(np.asarray(edge_u), dtype=np.int32)
            eb = np.ascontiguousarray(np.asarray(edge_b), dtype=np.int32)
            if eu.shape != eb.shape or eu.ndim != 1:
                raise ValueError('edge_u and edge_b must be 1-D arrays of equal length')
            rc = lib.blp_graph_create(int(n_users), int(n_biz), int(eu.size),
                                      eu.ctypes.data_as(ctypes.c_void_p),
                                      eb.ctypes.data_as(ctypes.c_void_p), int(device),
                                      ctypes.byref(self._h))
            _lib.check(rc, 'blp_graph_create')
        else:
            raise ValueError("build must be 'host' or 'device'")
        self.device = torch.device('cuda', int(device))
        self.n_users, self.n_biz = int(n_users), int(n_biz)
        # shared-id-space view (sorted id tables), None when built from local indices
        self.user_ids = None if user_ids is None else np.asarray(user_ids, dtype=np.int64)
        self.biz_ids = None if biz_ids is None else np.asarray(biz_ids, dtype=np.int64)
        self._deg = [None, None]

    # ------------------------------------------------------------------ construction
    @classmethod
    def from_id_edges(cls, ids_u, ids_b, device=None, build='device'):
        ids_u = np.asarray(ids_u, dtype=np.int64)
        ids_b = np.asarray(ids_b, dtype=np.int64)
        users, eu = np.unique(ids_u, return_inverse=True)
        bizs, eb = np.unique(ids_b, return_inverse=True)
        if users.size == 0:
            raise ValueError('empty edge list')
        if np.intersect1d(users, bizs, assume_unique=True).size:
            raise ValueError('graph is not bipartite by column: some id appears both as a user '
                             '(column 0) and as a business (column 1)')
        return cls(users.size, bizs.size, eu, eb, device=device, user_ids=users, biz_ids=bizs,
                   build=build)

    @classmethod
    def from_id_edges_device(cls, ids_u, ids_b, device=None):
        """The same for int64 CUDA tensors of shared-space ids: compaction (sorted id tables +
        inverse) and the disjointness check run on the device, the graph is built by
        ``blp_graph_create_device`` -- nothing but the two id tables visits the host."""
        dev = ids_u.device
        if ids_u.numel() == 0:
            raise ValueError('empty edge list')
        with torch.cuda.device(dev):
            users, eu = torch.unique(ids_u, return_inverse=True)
            bizs, eb = torch.unique(ids_b, return_inverse=True)
            pos = torch.searchsorted(bizs, users).clamp_(max=bizs.numel() - 1)
            if bool((bizs[pos] == users).any()):
                raise ValueError('graph is not bipartite by column: some id appears both as a user '
                                 '(column 0) and as a business (column 1)')
            return cls(int(users.numel()), int(bizs.numel()), eu.to(torch.int32), eb.to(torch.int32),
                       device=dev, user_ids=users.cpu().numpy(), biz_ids=bizs.cpu().numpy(),
                       build='device')

    @classmethod
    def from_edge_list(cls, path, src_col=0, dst_col=1, device=None, parse='device'):
        """``snap.LoadEdgeList(snap.PUNGraph, path, 0, 1)`` (similarity.py:16).  parse='device'
        (default): the text is parsed, compacted and turned into the CSR pair on the GPU;
        parse='host': pandas' C parser + the host-side compaction (same graph)."""
        if (src_col, dst_col) != (0, 1):
            raise ValueError('column 0 must hold users and column 1 businesses')
        if parse == 'device':
            u, b = read_edge_list_device(path, device)
            return cls.from_id_edges_device(u, b, device=device)
        if parse != 'host':
            raise ValueError("parse must be 'device' or 'host'")
        u, b = read_edge_list(path)
        return cls.from_id_edges(u, b, device=device)

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, '_h', None) is not None and self._h:
            self._lib.blp_graph_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ introspection
    def info(self):
        gi = _lib.GraphInfo()
        _lib.check(self._lib.blp_graph_info(self._h, ctypes.byref(gi)), 'blp_graph_info')
        return gi.as_dict()

    def degrees(self, side):
        """De-duplicated degrees of one side as a host int32 array (cached)."""
        if self._deg[side] is None:
            n = self.n_users if side == _lib.SIDE_USER else self.n_biz
            out = np.empty(n, dtype=np.int32)
            _lib.check(self._lib.blp_graph_degrees(self._h, side,
                                                   out.ctypes.data_as(ctypes.c_void_p)),
                       'blp_graph_degrees')
            self._deg[side] = out
        return self._deg[side]

    # ------------------------------------------------------------------ id space
    @staticmethod
    def _lookup(table, ids):
        ids = np.asarray(ids, dtype=np.int64)
        pos = np.searchsorted(table, ids)
        pos[pos >= table.size] = 0
        hit = table[pos] == ids
        return np.where(hit, pos, -1).astype(np.int32)

    def local_users(self, ids):
        """Shared-space ids -> local user indices, -1 where the id is not a user of the graph."""
        if self.user_ids is None:
            ids = np.asarray(ids, dtype=np.int64)
            return np.where((ids >= 0) & (ids < self.n_users), ids, -1).astype(np.int32)
        return self._lookup(self.user_ids, ids)

    def local_businesses(self, ids):
        if self.biz_ids is None:
            ids = np.asarray(ids, dtype=np.int64)
            return np.where((ids >= 0) & (ids < self.n_biz), ids, -1).astype(np.int32)
        return self._lookup(self.biz_ids, ids)

    # SNAP spellings used by the reference's set-level helpers ---------------------------
    def GetNI(self, nid):
        """``G.GetNI(i).GetDeg()`` (similarity.py:121) for an id of the shared id space."""
        u = int(self.local_users([nid])[0])
        if u >= 0 and self.degrees(_lib.SIDE_USER)[u] > 0:
            return _NodeIt(nid, int(self.degrees(_lib.SIDE_USER)[u]))
        b = int(self.local_businesses([nid])[0])
        if b >= 0 and self.degrees(_lib.SIDE_BUSINESS)[b] > 0:
            return _NodeIt(nid, int(self.degrees(_lib.SIDE_BUSINESS)[b]))
        raise RuntimeError('node %r is not in the graph' % (nid,))

    def Nodes(self):
        """``snap.Nodes(G)``: node iterators of every id with degree >= 1 (similarity.py:22)."""
        du, db = self.degrees(_lib.SIDE_USER), self.degrees(_lib.SIDE_BUSINESS)
        uid = self.user_ids if self.user_ids is not None else np.arange(self.n_users)
        bid = self.biz_ids if self.biz_ids is not None else np.arange(self.n_biz)
        for i in np.nonzero(du > 0)[0]:
            yield _NodeIt(int(uid[i]), int(du[i]))
        for i in np.nonzero(db > 0)[0]:
            yield _NodeIt(int(bid[i]), int(db[i]))

    def GetNodes(self):
        i = self.info()
        return i['n_users_in_graph'] + i['n_biz_in_graph']

    def GetEdges(self):
        return self.info()['n_edges']

    # ------------------------------------------------------------------ scoring
    def score_side(self, side, pair_u, pair_b, want=OUTPUTS_PER_SIDE, want_pa=False,
                   want_hop2=False, out=None, stream=None, out_ptr=None):
        """One ``blp_score_pairs`` call.  pair_u / pair_b: int32 CUDA tensors of local indices.

        Returns a dict of CUDA tensors (keys from ``want`` plus 'pa' / 'hop2' when asked).
        ``out`` may carry preallocated tensors under the same keys.  ``out_ptr`` maps keys to raw
        device addresses instead (n elements each, e.g. rows of a peer-mapped ``dist.ResultWindow``
        on another GPU): those columns are written there and are not part of the returned dict.
        """
        if not (pair_u.is_cuda and pair_b.is_cuda):
            raise ValueError('pair_u / pair_b must be CUDA tensors (use score_pairs_host for '
                             'host arrays)')
        if pair_u.dtype != torch.int32 or pair_b.dtype != torch.int32:
            raise ValueError('pair_u / pair_b must be int32')
        if pair_u.device != self.device or pair_b.device != self.device:
            raise ValueError('pairs live on %s, graph on %s' % (pair_u.device, self.device))
        pair_u, pair_b = pair_u.contiguous(), pair_b.contiguous()
        n = pair_u.numel()
        if pair_b.numel() != n:
            raise ValueError('pair_u and pair_b differ in length')
        dtypes = {'cn': torch.int32, 'union': torch.int32, 'jaccard': torch.float64,
                  'adamic': torch.float64, 'pa': torch.int64, 'hop2': torch.int32}
        keys = list(want) + (['pa'] if want_pa else []) + (['hop2'] if want_hop2 else [])
        raw = dict(out_ptr or {})
        if any(k not in dtypes for k in raw):
            raise ValueError('out_ptr keys must be among %s' % sorted(dtypes))
        res = {}
        for k in keys:
            if k in raw:
                continue
            t = None if out is None else out.get(k)
            if t is None:
                t = torch.empty(n, dtype=dtypes[k], device=self.device)
            elif t.dtype != dtypes[k] or t.numel() != n or not t.is_contiguous():
                raise ValueError('preallocated output %r has the wrong dtype/size' % k)
            res[k] = t

        def ptr(k):
            if k in raw:
                return ctypes.c_void_p(int(raw[k]))
            return ctypes.c_void_p(res[k].data_ptr()) if k in res else None

        if stream is None:
            stream = torch.cuda.current_stream(self.device)
        rc = self._lib.blp_score_pairs(self._h, int(side), ctypes.c_void_p(pair_u.data_ptr()),
                                       ctypes.c_void_p(pair_b.data_ptr()), n, ptr('cn'),
                                       ptr('union'), ptr('jaccard'), ptr('adamic'), ptr('pa'),
                                       ptr('hop2'), ctypes.c_void_p(stream.cuda_stream))
        _lib.check(rc, 'blp_score_pairs')
        return res

    def score_pairs(self, pair_u, pair_b, want_hop2=False, out=None, stream=None,
                    concurrent=True):
        """All seven reference outputs of every pair: u_cn,u_jaccard,u_adamic,b_cn,b_jaccard,
        b_adamic,pa (plus the two union sizes).  Device tensors in, device tensors out.

        With ``concurrent`` the business side is issued on a side stream (forked from and joined
        back to ``stream``), so its grouping kernels and the tails of both scoring grids overlap.
        """
        o_u = None if out is None else {k[2:]: v for k, v in out.items() if k.startswith('u_')}
        o_b = None if out is None else {k[2:]: v for k, v in out.items() if k.startswith('b_')}
        if out is not None and 'pa' in out:
            o_u['pa'] = out['pa']
        if stream is None:
            stream = torch.cuda.current_stream(self.device)
        if concurrent:
            # user side (the long one) on a high-priority stream, business side on a normal one:
            # the block scheduler serves the user grid first and lets the business grid fill in
            # as user CTAs retire, instead of the two grids stealing each other's SM slots
            if getattr(self, '_hi_stream', None) is None:
                self._hi_stream = torch.cuda.Stream(device=self.device, priority=-1)
                self._side_stream = torch.cuda.Stream(device=self.device)
            hi, side = self._hi_stream, self._side_stream
            hi.wait_stream(stream)
            side.wait_stream(stream)
            for which in 'bu':   # business side first: its short grid drains while users group
                if which == 'u':
                    with torch.cuda.stream(hi):
                        ru = self.score_side(_lib.SIDE_USER, pair_u, pair_b, want_pa=True,
                                             want_hop2=want_hop2, out=o_u, stream=hi)
                else:
                    with torch.cuda.stream(side):
                        rb = self.score_side(_lib.SIDE_BUSINESS, pair_u, pair_b,
                                             want_hop2=want_hop2, out=o_b, stream=side)
            for t in list(ru.values()) + list(rb.values()):
                t.record_stream(stream)
            stream.wait_stream(hi)
            stream.wait_stream(side)
        else:
            ru = self.score_side(_lib.SIDE_USER, pair_u, pair_b, want_pa=True,
                                 want_hop2=want_hop2, out=o_u, stream=stream)
            rb = self.score_side(_lib.SIDE_BUSINESS, pair_u, pair_b, want_hop2=want_hop2,
                                 out=o_b, stream=stream)
        res = {'u_' + k: v for k, v in ru.items() if k != 'pa'}
        res.update({'b_' + k: v for k, v in rb.items()})
        res['pa'] = ru['pa']
        return res

    def hop3_candidates(self, users, stream=None):
        """Businesses at BFS distance exactly 3 of every user (local indices; int32 CUDA tensor or
        array) -- make_examples' snap.GetNodesAtHop(G, u, 3, ...) (dataset_maker.py:137-139).
        Returns (offsets int64 [n+1], businesses int32 [total]) as CUDA tensors; the candidates
        of users[i] are businesses[offsets[i]:offsets[i+1]], ascending."""
        if not isinstance(users, torch.Tensor):
            users = torch.from_numpy(np.ascontiguousarray(users, dtype=np.int32))
        users = users.to(device=self.device, dtype=torch.int32).contiguous()
        n = users.numel()
        if stream is None:
            stream = torch.cuda.current_stream(self.device)
        sp = ctypes.c_void_p(stream.cuda_stream)
        with torch.cuda.device(self.device):
            counts = torch.zeros(n, dtype=torch.int64, device=self.device)
            _lib.check(self._lib.blp_hop3_count(self._h, ctypes.c_void_p(users.data_ptr()), n,
                                                ctypes.c_void_p(counts.data_ptr()), sp),
                       'blp_hop3_count')
            offsets = torch.zeros(n + 1, dtype=torch.int64, device=self.device)
            torch.cumsum(counts, 0, out=offsets[1:])
            total = int(offsets[-1].item())
            out = torch.empty(max(total, 1), dtype=torch.int32, device=self.device)
            _lib.check(self._lib.blp_hop3_fill(self._h, ctypes.c_void_p(users.data_ptr()), n,
                                               ctypes.c_void_p(offsets.data_ptr()),
                                               ctypes.c_void_p(out.data_ptr()), sp),
                       'blp_hop3_fill')
        return offsets, out[:total]

    def reserve_sms(self, n_sms):
        """Keep n_sms SMs out of the scoring grids (0 = use all); see blp_graph_reserve_sms."""
        _lib.check(self._lib.blp_graph_reserve_sms(self._h, int(n_sms)), 'blp_graph_reserve_sms')

    def score_stats(self, side):
        st = _lib.ScoreStats()
        _lib.check(self._lib.blp_score_stats(self._h, side, ctypes.byref(st)), 'blp_score_stats')
        return st.as_dict()

    def score_pairs_host(self, pair_u, pair_b, want_hop2=False):
        """Host arrays of LOCAL indices in, dict of host numpy arrays out (H2D + score + D2H)."""
        pu = torch.from_numpy(np.ascontiguousarray(pair_u, dtype=np.int32))
        pv = torch.from_numpy(np.ascontiguousarray(pair_b, dtype=np.int32))
        with torch.cuda.device(self.device):
            du = pu.to(self.device, non_blocking=False)
            dv = pv.to(self.device, non_blocking=False)
            res = self.score_pairs(du, dv, want_hop2=want_hop2)
            host = {k: v.cpu().numpy() for k, v in res.items()}
        return host

    def host_session(self, max_pairs, columns=None):
        """Reusable pinned/device buffers for repeated host-to-host scoring of <= max_pairs.
        columns: None = the seven reference outputs (48 B per pair come back), 'all' = plus the
        two union sizes (56 B), or an explicit tuple of column names."""
        return HostSession(self, max_pairs, columns=columns)

    def score_id_pairs(self, ids_u, ids_b, want_hop2=False):
        """Same, for ids of the reference's shared id space (unknown ids score 0)."""
        return self.score_pairs_host(self.local_users(ids_u), self.local_businesses(ids_b),
                                     want_hop2=want_hop2)


class HostSession(object):
    """End-to-end scoring with HOST buffers: page-locked pair and result arrays owned by the
    session, and ONE C-ABI call per step (`blp_score_pairs_host`) that uploads the ids, scores
    both sides and copies the result columns back, the copies overlapping the kernels inside the
    library.  By default the columns are the seven outputs the reference leaves on the host
    (similarity.py:61,106 + PA: 48 B per pair); the two union sizes are extra (``columns='all'``,
    56 B) -- the link is the bottleneck of this call, so bytes that nobody reads stay on the device.
    """

    ALL_KEYS = ('u_cn', 'u_union', 'u_jaccard', 'u_adamic', 'b_cn', 'b_union', 'b_jaccard',
                'b_adamic', 'pa')          # order of blp_score_pairs_host's output arguments
    REFERENCE_KEYS = ('u_cn', 'u_jaccard', 'u_adamic', 'b_cn', 'b_jaccard', 'b_adamic', 'pa')
    DTYPES = {'cn': torch.int32, 'union': torch.int32, 'jaccard': torch.float64,
              'adamic': torch.float64, 'pa': torch.int64}

    def __init__(self, graph, max_pairs, columns=None):
        self.g, self.n_max = graph, int(max_pairs)
        n = self.n_max
        if columns is None:
            columns = self.REFERENCE_KEYS
        elif columns == 'all':
            columns = self.ALL_KEYS
        bad = [c for c in columns if c not in self.ALL_KEYS]
        if bad:
            raise ValueError('unknown result columns %r' % (bad,))
        self.KEYS = tuple(k for k in self.ALL_KEYS if k in columns)
        self.h_u = torch.empty(n, dtype=torch.int32).pin_memory()
        self.h_b = torch.empty(n, dtype=torch.int32).pin_memory()
        self.h_out = {}
        for k in self.KEYS:
            self.h_out[k] = torch.empty(n, dtype=self.DTYPES[k.split('_')[-1]]).pin_memory()
        self.h2d_bytes_per_pair = 8
        self.d2h_bytes_per_pair = sum(self.h_out[k].element_size() for k in self.KEYS)

    def measure_link(self, n, reps=3):
        """The host link under this session's own buffers: pinned D2H of the result columns and
        H2D of the pair ids, timed alone.  The copy-back time is the floor under one step.
        OVERWRITES the session's pinned result buffers (call it before scoring, not after)."""
        n = min(int(n), self.n_max)
        dev = self.g.device
        with torch.cuda.device(dev):
            d = {k: torch.empty(n, dtype=self.h_out[k].dtype, device=dev) for k in self.KEYS}
            du = torch.empty(n, dtype=torch.int32, device=dev)
            best_d2h = best_h2d = float('inf')
            for _ in range(reps):
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                for k in self.KEYS:
                    self.h_out[k][:n].copy_(d[k], non_blocking=True)
                torch.cuda.synchronize(dev)
                best_d2h = min(best_d2h, time.perf_counter() - t0)
                t0 = time.perf_counter()
                du.copy_(self.h_u[:n], non_blocking=True)
                torch.cuda.synchronize(dev)
                best_h2d = min(best_h2d, time.perf_counter() - t0)
        d2h_bytes = self.d2h_bytes_per_pair * n
        return {'d2h_gbs': d2h_bytes / best_d2h / 1e9, 'h2d_gbs': 4 * n / best_h2d / 1e9,
                'd2h_floor_ms': best_d2h * 1e3,
                'what': 'pinned copies timed alone on this box; d2h_floor_ms = the %d result bytes '
                        'of one step at that rate' % d2h_bytes}

    def pinned_inputs(self, n):
        """Numpy views of the pinned pair buffers, for callers that fill them in place."""
        return self.h_u[:n].numpy(), self.h_b[:n].numpy()

    def score(self, pair_u, pair_b):
        """pair_u / pair_b: host int32 numpy arrays (local indices).  Returns {key: numpy view
        of the pinned result buffer} -- valid until the next call."""
        n = int(pair_u.size)
        if n > self.n_max or pair_b.size != n:
            raise ValueError('pair count %d exceeds the session capacity %d' % (n, self.n_max))
        hu, hb = self.pinned_inputs(n)
        hu[:] = pair_u
        hb[:] = pair_b
        return self.score_pinned(n)

    def score_pinned(self, n, user_chunks=0, lead_chunks=-1, biz_chunks=0):
        """Score the first n pairs already sitting in the pinned input buffers: ONE call of the
        C ABI's host-buffer entry point, blp_score_pairs_host (upload, both sides, copy-back, all
        overlapped inside the library; 0 / -1 / 0 select its default slice plan)."""
        n = int(n)
        if n > self.n_max:
            raise ValueError('pair count %d exceeds the session capacity %d' % (n, self.n_max))
        lib = self.g._lib
        outs = [self.h_out[k].data_ptr() if k in self.h_out else None for k in self.ALL_KEYS]
        _lib.check(lib.blp_score_pairs_host(self.g._h, self.h_u.data_ptr(), self.h_b.data_ptr(), n,
                                            *outs, int(user_chunks), int(lead_chunks),
                                            int(biz_chunks)), 'blp_score_pairs_host')
        return {k: self.h_out[k][:n].numpy() for k in self.KEYS}
