"""JSON helpers with the reference's on-disk formats (util.py:12-21 of the reference).

``examples.json``: ``{"<user>": {"<business>": 0|1}}``; score files: ``{"<user>": {"<business>": n}}``
-- whole-file JSON, string keys of the shared int id space, ints as bare ints and floats in
shortest-repr form (what ``json.dumps`` emits).
"""
import json


def load_json(fname):
    with open(fname) as fh:
        return json.load(fh)


def write_json(d, fname):
    with open(fname, 'w') as fh:
        fh.write(json.dumps(d))


# ---------------------------------------------------------------------------------------------
# The same two formats on the device (csrc/blp_json.cu): examples.json is parsed where the pairs
# are scored, and the score files are formatted there, byte for byte what write_json writes.
# ---------------------------------------------------------------------------------------------
CHUNK_BYTES = 64 << 20     # text produced, copied back and written per step


def _cuda_device(device):
    import torch
    if device is None:
        device = torch.cuda.current_device()
    return device if isinstance(device, torch.device) else torch.device('cuda', int(device))


def read_examples_device(fname, device=None):
    """``examples.json`` parsed ON the device (``blp_examples_count`` / ``blp_examples_parse``).

    Returns CUDA tensors ``(user_off, user_ids, biz_ids, labels)`` in file order -- int64
    ``[n_users + 1]`` (the pairs of user i are ``user_off[i]:user_off[i+1]``), int64 ``[n_users]``,
    int64 ``[n_pairs]``, int32 ``[n_pairs]`` -- or None when the file is outside the device grammar
    (what json.dumps writes for ``{"<u>": {"<b>": int}}``: canonical decimal keys, int32 labels,
    no duplicate keys); ``load_json`` is the reader for those."""
    import ctypes
    import numpy as np
    import torch
    from . import _lib
    lib = _lib.load()
    dev = _cuda_device(device)
    raw = np.fromfile(fname, dtype=np.uint8)
    with torch.cuda.device(dev):
        text = torch.from_numpy(raw).to(dev)
        st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        n_users, n_pairs = ctypes.c_int64(0), ctypes.c_int64(0)
        rc = lib.blp_examples_count(ctypes.c_void_p(text.data_ptr()), int(text.numel()),
                                    ctypes.byref(n_users), ctypes.byref(n_pairs), st)
        if rc == _lib.BLP_ERR_UNSUPPORTED:
            return None
        _lib.check(rc, 'blp_examples_count')
        nu, npairs = int(n_users.value), int(n_pairs.value)
        user_off = torch.empty(nu + 1, dtype=torch.int64, device=dev)
        user_ids = torch.empty(nu, dtype=torch.int64, device=dev)
        biz_ids = torch.empty(npairs, dtype=torch.int64, device=dev)
        labels = torch.empty(npairs, dtype=torch.int32, device=dev)
        rc = lib.blp_examples_parse(ctypes.c_void_p(text.data_ptr()), int(text.numel()), nu, npairs,
                                    *[ctypes.c_void_p(t.data_ptr()) for t in (user_off, user_ids, biz_ids, labels)],
                                    st)
        if rc == _lib.BLP_ERR_UNSUPPORTED:     # duplicate keys
            return None
        _lib.check(rc, 'blp_examples_parse')
    return user_off, user_ids, biz_ids, labels


def write_scores_json_device(fname, user_off, user_ids, biz_ids, in_graph, values=None, kind=None,
                             chunk_bytes=CHUNK_BYTES, buffers=None, stats=None):
    """One score file from CUDA tensors, byte for byte what ``write_json`` writes for the dict
    ``similarity._emit`` builds: ``{"<u>": {"<b>": v}}`` over the example users in order.

    ``user_off`` / ``user_ids`` / ``biz_ids`` as ``read_examples_device`` returns them, ``in_graph``
    a bool / uint8 tensor per pair (False: written as the int 0), ``values`` the pair's column of
    type ``kind`` (``_lib.JSON_*``), or None to write only the out-of-graph zeros.  The text is
    made in chunks of at most ``chunk_bytes`` (or one user's text, if longer) cut at user
    boundaries, each copied into one page-locked buffer and appended to the file.  ``buffers``: a
    dict the caller keeps to reuse the staging buffers across files.  ``stats``: a dict in which
    the CUDA-event times of the format kernels ('format_ms') and of the copies ('d2h_ms') and the
    host time of the file writes ('write_s') are accumulated."""
    import ctypes
    import time
    import numpy as np
    import torch
    from . import _lib
    lib = _lib.load()
    dev = user_ids.device
    n_users = int(user_ids.numel())
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        st = ctypes.c_void_p(stream.cuda_stream)
        in_graph = in_graph.to(torch.uint8).contiguous()
        if values is None:
            kind = _lib.JSON_INT32
        else:
            values = values.contiguous()
        args = [ctypes.c_void_p(user_off.data_ptr()), ctypes.c_void_p(user_ids.data_ptr()), n_users,
                ctypes.c_void_p(biz_ids.data_ptr()), ctypes.c_void_p(in_graph.data_ptr()),
                ctypes.c_void_p(values.data_ptr() if values is not None else None), int(kind)]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if stats is not None else None

        def mark(i):
            if ev is not None:
                ev[i].record(stream)

        def add(key, value):
            if stats is not None:
                stats[key] = stats.get(key, 0.0) + value

        lengths = torch.empty(n_users, dtype=torch.int64, device=dev)
        mark(0)
        _lib.check(lib.blp_json_scores_count(*args, ctypes.c_void_p(lengths.data_ptr()), st),
                   'blp_json_scores_count')
        text_off = torch.zeros(n_users + 1, dtype=torch.int64, device=dev)
        torch.cumsum(lengths, 0, out=text_off[1:])
        mark(1)
        off = text_off.cpu().numpy()
        if ev is not None:
            add('format_ms', ev[0].elapsed_time(ev[1]))
        with open(fname, 'wb') as fh:
            if off[-1] == 0:
                fh.write(b'{}')
                return
            cap = max(int(chunk_bytes), int(np.diff(off).max()))
            buffers = {} if buffers is None else buffers
            if buffers.get('cap', 0) < cap or buffers.get('device') != dev:
                buffers.update(cap=cap, device=dev, dev=torch.empty(cap, dtype=torch.uint8, device=dev),
                               host=torch.empty(cap, dtype=torch.uint8).pin_memory())
            dbuf, hbuf = buffers['dev'], buffers['host']
            fh.write(b'{')
            skip, begin = 2, 0     # the first user's text starts with the ", " of a later one
            while begin < n_users:
                end = max(int(np.searchsorted(off, off[begin] + cap, side='right')) - 1, begin + 1)
                nbytes = int(off[end] - off[begin])
                mark(0)
                _lib.check(lib.blp_json_scores_fill(*args, ctypes.c_void_p(text_off.data_ptr()), begin, end,
                                                    ctypes.c_void_p(dbuf.data_ptr()), st),
                           'blp_json_scores_fill')
                mark(1)
                hbuf[:nbytes].copy_(dbuf[:nbytes], non_blocking=True)
                mark(2)
                stream.synchronize()
                if ev is not None:
                    add('format_ms', ev[0].elapsed_time(ev[1]))
                    add('d2h_ms', ev[1].elapsed_time(ev[2]))
                t0 = time.perf_counter()
                fh.write(hbuf[skip:nbytes].numpy())
                add('write_s', time.perf_counter() - t0)
                skip, begin = 0, end
            fh.write(b'}')


def write_edge_list(fname, ids_u, ids_b):
    """``graph.txt``: one "<user_id> <business_id>" line per review (dataset_maker.py:197)."""
    import numpy as np
    arr = np.stack([np.asarray(ids_u, dtype=np.int64), np.asarray(ids_b, dtype=np.int64)], axis=1)
    np.savetxt(fname, arr, fmt='%d %d')


# ---------------------------------------------------------------------------------------------
# Columnar sidecar (SURVEY.md section 8f, rank 3).  Nested JSON is tens of GB of text at 100M
# pairs; the same information as three flat arrays in an .npz is 16-20 B per pair and loads
# without parsing.  The JSON format stays the interchange format of the reference's readers
# (eval.py:14, supervised_models.py:81-86); these two functions convert losslessly both ways.
# ---------------------------------------------------------------------------------------------
def write_pairs_npz(fname, ids_u, ids_b, values):
    """One score (or label) file as columns: user id, business id, value.  Integer-valued files
    (cn, labels, literal zeros) are stored as int64, everything else as float64."""
    import numpy as np
    v = np.asarray(values)   # floats that happen to be whole stay float: jaccard 0.0 is not int 0
    np.savez(fname, u=np.asarray(ids_u, dtype=np.int64), b=np.asarray(ids_b, dtype=np.int64), v=v)


def read_pairs_npz(fname):
    import numpy as np
    z = np.load(fname)
    return z['u'], z['b'], z['v']


def dict_to_columns(d):
    """{"<u>": {"<b>": x}} -> (ids_u, ids_b, values, int_mask): int_mask remembers which values
    were Python ints (the reference mixes int 0 and floats in one file, similarity.py:59-60,118)."""
    import numpy as np
    us, bs, vs, im = [], [], [], []
    for u, row in d.items():
        for b, x in row.items():
            us.append(int(u))
            bs.append(int(b))
            vs.append(float(x))
            im.append(isinstance(x, int))
    return (np.asarray(us, dtype=np.int64), np.asarray(bs, dtype=np.int64),
            np.asarray(vs, dtype=np.float64), np.asarray(im, dtype=bool))


def columns_to_dict(ids_u, ids_b, values, int_mask=None):
    """Inverse of dict_to_columns: the nested dict json.dumps turns into the reference's file."""
    import numpy as np
    v = np.asarray(values)
    ints = v.dtype.kind in 'iu'
    out = {}
    im = None if int_mask is None else np.asarray(int_mask, dtype=bool).tolist()
    for i, (u, b, x) in enumerate(zip(np.asarray(ids_u).tolist(), np.asarray(ids_b).tolist(),
                                      v.tolist())):
        if ints or (im is not None and im[i]):
            x = int(x)
        out.setdefault(str(u), {})[str(b)] = x
    return out


def json_to_npz(json_file, npz_file):
    import numpy as np
    u, b, v, im = dict_to_columns(load_json(json_file))
    np.savez(npz_file, u=u, b=b, v=v, int_mask=im)


def npz_to_json(npz_file, json_file):
    import numpy as np
    z = np.load(npz_file)
    write_json(columns_to_dict(z['u'], z['b'], z['v'], z['int_mask'] if 'int_mask' in z else None),
               json_file)
