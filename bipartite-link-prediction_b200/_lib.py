"""ctypes binding of the C ABI in include/blp.h, plus the in-tree nvcc build recipe.

There is no fallback: if libblp.so is missing or a symbol cannot be bound the import of the
scoring path raises, and every compute entry point fails without a CUDA device.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, 'csrc')
INCLUDE = os.path.join(_ROOT, 'include')
LIB_PATH = os.path.join(_HERE, 'libblp.so')
if os.environ.get('BLP_LIB_PATH'):        # developer override: A/B a prebuilt variant (tools/build_variants.py)
    LIB_PATH = os.path.abspath(os.environ['BLP_LIB_PATH'])
SOURCES = ('blp_graph.cu', 'blp_build.cu', 'blp_score.cu', 'blp_host.cu', 'blp_hop3.cu', 'blp_eval.cu',
           'blp_peer.cu')

BLP_OK = 0
BLP_ERR_INVALID, BLP_ERR_CUDA, BLP_ERR_OOM, BLP_ERR_RANGE, BLP_ERR_UNSUPPORTED = -1, -2, -3, -4, -5
SIDE_USER, SIDE_BUSINESS = 0, 1
PATH_GROUPED, PATH_BIZ_INDEX = 0, 1     # blp_score_stats_t.path

# every symbol include/blp.h declares
EXPORTS = ('blp_version', 'blp_last_error', 'blp_device_count', 'blp_graph_create',
           'blp_graph_destroy', 'blp_graph_info', 'blp_graph_degrees', 'blp_score_pairs',
           'blp_score_stats', 'blp_graph_reserve_sms', 'blp_graph_create_device',
           'blp_hop3_count', 'blp_hop3_fill', 'blp_eval_precision_at_k', 'blp_eval_roc_auc',
           'blp_score_pairs_host', 'blp_peer_alloc', 'blp_peer_open', 'blp_peer_close',
           'blp_peer_free', 'blp_derive_pairs', 'blp_peer_push', 'blp_edge_list_count',
           'blp_edge_list_parse')
IPC_HANDLE_BYTES = 64


class GraphInfo(ctypes.Structure):
    _fields_ = [('n_users', ctypes.c_int32), ('n_biz', ctypes.c_int32),
                ('n_edges_in', ctypes.c_int64), ('n_edges', ctypes.c_int64),
                ('n_users_in_graph', ctypes.c_int32), ('n_biz_in_graph', ctypes.c_int32),
                ('max_user_degree', ctypes.c_int32), ('max_biz_degree', ctypes.c_int32),
                ('device_bytes', ctypes.c_int64), ('device', ctypes.c_int32),
                ('sm_count', ctypes.c_int32), ('n_hub_biz', ctypes.c_int32),
                ('n_hub_users', ctypes.c_int32), ('hub_min_biz_degree', ctypes.c_int32),
                ('hub_min_user_degree', ctypes.c_int32), ('biz_index_bytes', ctypes.c_int64),
                ('biz_index_build_ms', ctypes.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ScoreStats(ctypes.Structure):
    _fields_ = [('n_pairs', ctypes.c_int64), ('n_groups', ctypes.c_int64),
                ('kernel_launches', ctypes.c_int32), ('ctas', ctypes.c_int32),
                ('threads_per_cta', ctypes.c_int32), ('smem_bytes', ctypes.c_int32),
                ('range_passes', ctypes.c_int32), ('group_ms', ctypes.c_float),
                ('score_ms', ctypes.c_float), ('light_ms', ctypes.c_float),
                ('light_groups', ctypes.c_int32), ('path', ctypes.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def nvcc_command(out=LIB_PATH, extra=()):
    nvcc = os.environ.get('NVCC', 'nvcc')
    return [nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
            '-Xcompiler', '-fPIC', '-shared', '-I', INCLUDE, *extra,
            *[os.path.join(CSRC, s) for s in SOURCES], '-o', out]


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, 'blp.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile the CUDA extension in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    cmd = nvcc_command(extra=('-Xptxas', '-v') if verbose else ())
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + ' '.join(cmd) + '\n' + res.stdout)
    if verbose:
        print(res.stdout)
    return LIB_PATH


_lib = None


def load():
    """dlopen libblp.so and bind every exported symbol; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'CUDA extension %s is not built; run `python -c "import __graft_entry__ as g; '
            'g.build()"` (there is no CPU fallback)' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise RuntimeError('libblp.so does not export %s' % name)
    i32p, i64p, f64p = (ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64),
                        ctypes.POINTER(ctypes.c_double))
    lib.blp_version.restype = ctypes.c_int
    lib.blp_last_error.restype = ctypes.c_char_p
    lib.blp_device_count.argtypes = [ctypes.POINTER(ctypes.c_int)]
    lib.blp_graph_create.argtypes = [ctypes.c_int32, ctypes.c_int32, ctypes.c_int64,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                     ctypes.POINTER(ctypes.c_void_p)]
    lib.blp_graph_create_device.argtypes = [ctypes.c_int32, ctypes.c_int32, ctypes.c_int64,
                                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                            ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]
    lib.blp_hop3_count.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                   ctypes.c_void_p, ctypes.c_void_p]
    lib.blp_hop3_fill.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                  ctypes.c_void_p, ctypes.c_void_p]
    lib.blp_eval_precision_at_k.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                            ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p,
                                            ctypes.c_void_p]
    lib.blp_eval_roc_auc.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                     ctypes.POINTER(ctypes.c_uint64), ctypes.c_void_p]
    lib.blp_graph_destroy.argtypes = [ctypes.c_void_p]
    lib.blp_graph_info.argtypes = [ctypes.c_void_p, ctypes.POINTER(GraphInfo)]
    lib.blp_graph_degrees.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    lib.blp_score_pairs.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                    ctypes.c_void_p, ctypes.c_int64] + [ctypes.c_void_p] * 7
    lib.blp_score_pairs_host.argtypes = ([ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_int64] + [ctypes.c_void_p] * 9 + [ctypes.c_int] * 3)
    lib.blp_score_stats.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ScoreStats)]
    lib.blp_graph_reserve_sms.argtypes = [ctypes.c_void_p, ctypes.c_int]
    lib.blp_peer_alloc.argtypes = [ctypes.c_int, ctypes.c_int64, ctypes.POINTER(ctypes.c_void_p),
                                   ctypes.c_char_p]
    lib.blp_peer_open.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.POINTER(ctypes.c_void_p)]
    lib.blp_peer_close.argtypes = [ctypes.c_int, ctypes.c_void_p]
    lib.blp_peer_free.argtypes = [ctypes.c_int, ctypes.c_void_p]
    lib.blp_edge_list_count.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.POINTER(ctypes.c_int64), ctypes.c_void_p]
    lib.blp_edge_list_parse.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_void_p]
    lib.blp_peer_push.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    lib.blp_derive_pairs.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64] + \
        [ctypes.c_void_p] * 8
    for name in EXPORTS:
        if name not in ('blp_last_error',):
            getattr(lib, name).restype = ctypes.c_int
    del i32p, i64p, f64p
    _lib = lib
    return lib


def check(rc, what):
    """Map a negative blp_status to the Python exception the host layer promises."""
    if rc == BLP_OK:
        return
    msg = load().blp_last_error().decode('utf-8', 'replace')
    text = '%s failed (%d): %s' % (what, rc, msg)
    if rc in (BLP_ERR_INVALID, BLP_ERR_RANGE):
        raise ValueError(text)
    if rc == BLP_ERR_OOM:
        raise MemoryError(text)
    raise RuntimeError(text)
