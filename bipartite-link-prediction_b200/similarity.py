"""Drop-in for the reference's ``similarity.py``: same six call signatures, same file formats.

    main(example_file, graph_file, u_methods, u_outfiles, b_methods, b_outfiles)  similarity.py:11
    users(examples, G, methods, outfiles)                                          similarity.py:20
    business(examples, G, methods, outfiles)                                       similarity.py:63
    jaccard(setone, settwo)                                                        similarity.py:108
    common_neighbors(setone, settwo)                                               similarity.py:113
    adamic_adar(setone, settwo, G)                                                 similarity.py:116
    preferential_attachment(setone, settwo)      (no Python original; "Link prediction.R":400-415)

``examples`` is the reference's ``{"<user>": {"<business>": 0|1}}`` dict (dataset_maker.py:142-159),
``G`` is a ``BipartiteGraph`` (what ``LoadEdgeList`` below returns), score files are
``{"<user>": {"<business>": score}}`` with the key set of ``examples`` (similarity.py:49-61), read
unchanged by eval.py:14-18, supervised_models.py:81-86 and supervised_classifier.py:23-25.

``users`` / ``business`` flatten the examples into pair arrays and make ONE call per side into
the CUDA library (``blp_score_pairs``), which yields all three methods at once; the per-method
loop only selects which array is written where.  ``main`` keeps the whole step on the device when
``examples.json`` is in the device reader's grammar (what json.dumps writes for the reference's
dict): the file is parsed there, scored, and every score file is formatted there, byte for byte
what ``users`` / ``business`` write; any other file goes through ``json.load`` and those two.  The three set-level helpers keep their
reference meaning on Python sets -- they are the public formulas, not the bulk path.
"""
import math
from collections import defaultdict

import numpy as np

from . import _lib, util
from .graph import BipartiteGraph

METHODS = ('common_neighbors', 'jaccard', 'adamic_adar', 'preferential_attachment')
_COLUMN = {'common_neighbors': 'cn', 'jaccard': 'jaccard', 'adamic_adar': 'adamic',
           'preferential_attachment': 'pa'}
# how _emit types each column in the file: cn / pa as ints, jaccard as floats, adamic as floats
# except its untouched int 0
_KIND = {'cn': _lib.JSON_INT32, 'pa': _lib.JSON_INT64, 'jaccard': _lib.JSON_FLOAT64,
         'adamic': _lib.JSON_FLOAT64_INT_ZERO}

PUNGraph = 'PUNGraph'   # placeholder for snap.PUNGraph in LoadEdgeList(PUNGraph, file, 0, 1)


def LoadEdgeList(graph_type, graph_file, src_col=0, dst_col=1, device=None):
    """``snap.LoadEdgeList(snap.PUNGraph, graph_file, 0, 1)`` (similarity.py:16)."""
    return BipartiteGraph.from_edge_list(graph_file, src_col, dst_col, device=device)


def main(example_file, graph_file, u_methods, u_outfiles, b_methods, b_outfiles, *,
         device=None, reproduce_reference_bug=False, sidecar=False):
    ex = util.read_examples_device(example_file, device)
    if ex is None:   # outside the device reader's grammar: json.load decides what the file means
        examples = util.load_json(example_file)
        G = LoadEdgeList(PUNGraph, graph_file, 0, 1, device=device)
        users(examples, G, u_methods, u_outfiles, sidecar=sidecar)
        business(examples, G, b_methods, b_outfiles, reproduce_reference_bug=reproduce_reference_bug,
                 sidecar=sidecar)
        return G
    G = LoadEdgeList(PUNGraph, graph_file, 0, 1, device=device)
    skip = ('adamic_adar',) if reproduce_reference_bug else ()
    _main_device(G, ex, [(_lib.SIDE_USER, u_methods, u_outfiles, ()),
                         (_lib.SIDE_BUSINESS, b_methods, b_outfiles, skip)], sidecar)
    return G


def _lookup_device(table, ids):
    """BipartiteGraph._lookup on the device: local index of every id, -1 where it is not in table."""
    import torch
    t = torch.from_numpy(table).to(ids.device)
    pos = torch.searchsorted(t, ids).clamp_(max=t.numel() - 1)
    return torch.where(t[pos] == ids, pos, -1).to(torch.int32)


def _device_pairs(G, ex):
    """Example arrays of read_examples_device -> (user_off, user_ids, biz_ids, per-pair user ids,
    local user / business indices, in-graph mask), as _flatten + _score_side make them."""
    import torch
    dev = G.device
    with torch.cuda.device(dev):
        user_off, user_ids, biz_ids, _ = (t.to(dev) for t in ex)
        ids_u = torch.repeat_interleave(user_ids, user_off[1:] - user_off[:-1],
                                        output_size=biz_ids.numel())
        lu, lb = _lookup_device(G.user_ids, ids_u), _lookup_device(G.biz_ids, biz_ids)
        du = torch.from_numpy(G.degrees(_lib.SIDE_USER)).to(dev)
        db = torch.from_numpy(G.degrees(_lib.SIDE_BUSINESS)).to(dev)
        in_graph = ((lu >= 0) & (lb >= 0) & (du[lu.clamp(min=0).long()] > 0) &
                    (db[lb.clamp(min=0).long()] > 0))
    return user_off, user_ids, biz_ids, ids_u, lu, lb, in_graph


def _write_side(pairs, res, methods, outfiles, skip=(), sidecar=False, buffers=None, stats=None):
    """_emit's loop with the device formatter: one file per (method, file), from one side's
    scores `res` (G.score_side's dict)."""
    user_off, user_ids, biz_ids, ids_u, _, _, in_graph = pairs
    for m, f in zip(methods, outfiles):
        col = _COLUMN.get(m)
        vals = None if col is None or m in skip else res[col]
        util.write_scores_json_device(f, user_off, user_ids, biz_ids, in_graph, vals, _KIND.get(col),
                                      buffers=buffers, stats=stats)
        if sidecar:
            _save_sidecar(f, *_sidecar_columns(ids_u, biz_ids, in_graph, vals, col))


def _main_device(G, ex, sides, sidecar):
    import torch
    pairs = _device_pairs(G, ex)
    _, _, _, _, lu, lb, _ = pairs
    buffers = {}
    with torch.cuda.device(G.device):
        for side, methods, outfiles, skip in sides:
            res = G.score_side(side, lu, lb, want_pa=True)
            _write_side(pairs, res, methods, outfiles, skip, sidecar, buffers)


def _sidecar_columns(ids_u, biz_ids, in_graph, vals, col):
    """util.dict_to_columns of the dict _emit builds, computed from the pair arrays."""
    import torch
    if vals is None:                 # only the out-of-graph zeros
        keep = ~in_graph
        v = torch.zeros_like(ids_u, dtype=torch.float64)
        im = torch.ones_like(in_graph)
    else:
        keep = torch.ones_like(in_graph)
        v = torch.where(in_graph, vals.to(torch.float64), 0.0)
        im = ~in_graph
        if col in ('cn', 'pa'):
            im = torch.ones_like(in_graph)
        elif col == 'adamic':
            im = im | (vals == 0)
    return tuple(t[keep].cpu().numpy() for t in (ids_u, biz_ids, v, im))


def _save_sidecar(f, u, b, v, im):
    # columnar copy beside the JSON (SURVEY 8f rank 3); same content, no parsing
    np.savez(f[:-5] + '.npz' if f.endswith('.json') else f + '.npz', u=u, b=b, v=v, int_mask=im)


def _flatten(examples):
    us, bs = [], []
    for u in examples:
        for v in examples[u]:
            us.append(u)
            bs.append(v)
    ids_u = np.fromiter((int(u) for u in us), dtype=np.int64, count=len(us))
    ids_b = np.fromiter((int(b) for b in bs), dtype=np.int64, count=len(bs))
    return us, bs, ids_u, ids_b


def _score_side(G, side, ids_u, ids_b):
    import torch
    lu, lb = G.local_users(ids_u), G.local_businesses(ids_b)
    du = G.degrees(_lib.SIDE_USER)
    db = G.degrees(_lib.SIDE_BUSINESS)
    in_graph = (lu >= 0) & (lb >= 0)
    in_graph[in_graph] &= (du[lu[in_graph]] > 0) & (db[lb[in_graph]] > 0)
    with torch.cuda.device(G.device):
        tu = torch.from_numpy(lu).to(G.device)
        tb = torch.from_numpy(lb).to(G.device)
        res = G.score_side(side, tu, tb, want_pa=True)
        host = {k: v.cpu().numpy() for k, v in res.items()}
    return host, in_graph


def _emit(examples, keys_u, keys_b, host, in_graph, methods, outfiles, skip_in_graph=(),
          sidecar=False):
    out = []
    for m, f in zip(methods, outfiles):
        sim = defaultdict(dict)
        col = _COLUMN.get(m)
        if col is None:
            # unknown method name: the reference writes only the literal zeros (similarity.py:53-60)
            for i, (u, v) in enumerate(zip(keys_u, keys_b)):
                if not in_graph[i]:
                    sim[u][v] = 0
        else:
            vals = host[col].tolist()
            is_float = col in ('jaccard', 'adamic')
            for i, (u, v) in enumerate(zip(keys_u, keys_b)):
                if not in_graph[i]:
                    sim[u][v] = 0                       # similarity.py:59-60, 104-105
                elif m in skip_in_graph:
                    continue
                elif is_float and not (col == 'adamic' and vals[i] == 0.0):
                    sim[u][v] = float(vals[i])
                else:
                    sim[u][v] = int(vals[i])            # cn, pa, and adamic's untouched int 0
        util.write_json(sim, f)
        if sidecar:
            _save_sidecar(f, *util.dict_to_columns(sim))
        out.append(sim)
    return out


def users(examples, G, methods, outfiles, *, sidecar=False):
    keys_u, keys_b, ids_u, ids_b = _flatten(examples)
    host, in_graph = _score_side(G, _lib.SIDE_USER, ids_u, ids_b)
    return _emit(examples, keys_u, keys_b, host, in_graph, methods, outfiles, sidecar=sidecar)


def business(examples, G, methods, outfiles, *, reproduce_reference_bug=False, sidecar=False):
    """``reproduce_reference_bug=True`` omits in-graph ``adamic_adar`` entries exactly as the
    reference's mistyped branch does (similarity.py:102); the default writes the intended score
    (similarity.py:103)."""
    keys_u, keys_b, ids_u, ids_b = _flatten(examples)
    host, in_graph = _score_side(G, _lib.SIDE_BUSINESS, ids_u, ids_b)
    skip = ('adamic_adar',) if reproduce_reference_bug else ()
    return _emit(examples, keys_u, keys_b, host, in_graph, methods, outfiles, skip_in_graph=skip,
                 sidecar=sidecar)


# ----------------------------------------------------------------------------- set-level API
def jaccard(setone, settwo):
    inter = len(setone & settwo)
    return float(inter) / float(len(setone) + len(settwo) - inter)


def common_neighbors(setone, settwo):
    return len(setone & settwo)


def adamic_adar(setone, settwo, G):
    total = 0
    for i in setone & settwo:
        deg = G.GetNI(i).GetDeg()
        if deg > 1:
            total += (math.log(deg)) ** -1      # the reference's exact expression (similarity.py:123)
    return total


def preferential_attachment(setone, settwo):
    return len(setone) * len(settwo)


if __name__ == '__main__':   # same literal paths as similarity.py:128-142
    for split in ('train', 'test'):
        d = './data/%s/' % split
        main(d + 'examples.json', d + 'graph.txt',
             ['common_neighbors', 'jaccard', 'adamic_adar'],
             [d + 'u_cn.json', d + 'u_jaccard.json', d + 'u_adamic.json'],
             ['common_neighbors', 'jaccard', 'adamic_adar'],
             [d + 'b_cn.json', d + 'b_jaccard.json', d + 'b_adamic.json'])
