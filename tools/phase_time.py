"""Developer tool: per-phase cycle shares of the CTA kernel (k_score_side) from a BLP_PHASE_TIMING
build of the SAME sources (compiled into variants/libblp_phase.so on first use).  Thread 0 of every
CTA adds clock64() deltas at the phase boundaries to a global table; the shares are of CTA-resident
cycles.  Writes gpurun_out/phase_<config>.json (copy to profiles/r02_phase_shares.json for bench.py).
usage: phase_time.py [CONFIG] [n_pairs]"""
import ctypes, importlib, json, os, subprocess, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
L = importlib.import_module('bipartite-link-prediction_b200._lib')
out = os.path.join(ROOT, 'bipartite-link-prediction_b200', 'variants', 'libblp_phase.so')
if not os.path.exists(out):
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(L.nvcc_command(out=out, extra=('-DBLP_PHASE_TIMING',)), check=True)
L.LIB_PATH = out
graph = importlib.import_module('bipartite-link-prediction_b200.graph')
synth = importlib.import_module('bipartite-link-prediction_b200.synth')
cfgname = sys.argv[1] if len(sys.argv) > 1 else 'C2'
cfg, eu, eb, pu, pv = synth.make_config(cfgname, n_pairs=int(sys.argv[2]) if len(sys.argv) > 2 else None)
G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, device=0)
lib = L.load()
lib.blp_debug_phase_cycles.argtypes = [ctypes.c_void_p, ctypes.c_int]
du, dv = torch.from_numpy(pu).cuda(), torch.from_numpy(pv).cuda()
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
names = ['fetch(top barrier..item)', 'exp tile load+scan', 'clear / hub-bitmap copy+OR', 'SET sweep', '-',
         'hop2 finalize', 'pair tile load+scan', 'TEST sweep', 'epilogue + bitmap clear']
buf = (ctypes.c_ulonglong * 16)()
doc = {'config': cfgname, 'pairs': int(pu.size), 'sides': {}}
for side, tag in ((0, 'user'), (1, 'business')):
    G.score_side(side, du, dv, want_pa=(side == 0))
    lib.blp_debug_phase_cycles(buf, 1)
    flush.zero_()
    G.score_side(side, du, dv, want_pa=(side == 0))
    lib.blp_debug_phase_cycles(buf, 1)
    st = G.score_stats(side)
    tot = float(sum(buf[:9]))
    shares = {n: buf[i] / tot for i, n in enumerate(names) if n != '-'}
    print('side', side, 'score_ms %.3f' % st['score_ms'], 'light_ms %.3f' % st['light_ms'], 'ctas', st['ctas'],
          'sum cycles/cta %.3g' % (tot / st['ctas']))
    for n, v in shares.items():
        print('   %-28s %5.1f%%' % (n, 100.0 * v))
    doc['sides'][tag] = {'score_ms_instrumented': st['score_ms'], 'light_ms': st['light_ms'], 'ctas': st['ctas'],
                         'groups': st['n_groups'], 'light_groups': st['light_groups'], 'shares': shares}
u = doc['sides']['user']['shares']
doc['intersection_share_of_user_side'] = u['pair tile load+scan'] + u['TEST sweep'] + u['epilogue + bitmap clear']
doc['expansion_share_of_user_side'] = (u['exp tile load+scan'] + u['clear / hub-bitmap copy+OR'] + u['SET sweep'] +
                                       u['hop2 finalize'])
doc['source'] = ('tools/phase_time.py on a -DBLP_PHASE_TIMING build of the shipped kernels: clock64() deltas of '
                 'thread 0 of every k_score_side CTA, user side of %s; intersection = pair tile load + TEST sweep '
                 '+ epilogue.  The warp-per-group kernel beside it is not instrumented; the CTA kernel is the '
                 'critical path of the user side, its share is applied to the whole span' % cfgname)
os.makedirs(os.path.join(ROOT, 'gpurun_out'), exist_ok=True)
with open(os.path.join(ROOT, 'gpurun_out', 'phase_%s.json' % cfgname), 'w') as fh:
    json.dump(doc, fh, indent=1)
