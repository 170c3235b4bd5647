"""Developer tool: the probe path of the intersection (small hop-2 list against the partner's
bitmap) on and off, same box, same process.  Times both sides per setting and checks that every
output column is bit-identical to the path-off run.
usage: probe_ab.py [CONFIG] [PAIRS] -- settings come from BLP_AB_SETTINGS
       ("min_deg:ratio:light:one_hub_groups,..."; min_deg 0 = probe path off, -1 = library default; light 0/1 = the
       warp-per-group kernel off/on)."""
import importlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
graph = importlib.import_module('bipartite-link-prediction_b200.graph')
synth = importlib.import_module('bipartite-link-prediction_b200.synth')

name = sys.argv[1] if len(sys.argv) > 1 else 'C2'
n_pairs = int(sys.argv[2]) if len(sys.argv) > 2 else None
settings = os.environ.get('BLP_AB_SETTINGS', '0:2:0:0,-1:2:1:0,-1:2:1:1,-1:1:1:1,-1:4:1:1,256:2:1:1')
cfg, eu, eb, pu, pv = synth.make_config(name, n_pairs=n_pairs)
du, dv = torch.from_numpy(pu).cuda(), torch.from_numpy(pv).cuda()
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
base = None
for s in settings.split(','):
    min_deg, ratio, light, medium = s.split(':')[:4]
    extra = s.split(':')[4:5]         # optional: hub_min_deg
    os.environ.pop('BLP_HUB_MIN_DEG', None)
    if extra and int(extra[0]) > 0:
        os.environ['BLP_HUB_MIN_DEG'] = extra[0]
    os.environ['BLP_LIGHT'] = light
    os.environ['BLP_LIGHT_HUBS'] = medium
    os.environ.pop('BLP_PROBE_MIN_DEG', None)
    if int(min_deg) >= 0:
        os.environ['BLP_PROBE_MIN_DEG'] = min_deg
    os.environ['BLP_PROBE_RATIO'] = ratio
    G = graph.BipartiteGraph(cfg['n_users'], cfg['n_biz'], eu, eb, device=0)
    info = G.info()
    res, outs, lms = [], [], []
    for side in (0, 1):
        ms, out = [], None
        for it in range(7):
            flush.zero_()
            out = G.score_side(side, du, dv, want_pa=(side == 0), out=out)
            torch.cuda.synchronize()
            ms.append(G.score_stats(side)['score_ms'])
        res.append(min(ms[1:]))
        lms.append(G.score_stats(side)['light_ms'])
        outs.append({k: v.clone() for k, v in out.items()})
    same = ''
    if base is None:
        base = outs
    else:
        bad = [(sd, k) for sd in (0, 1) for k in outs[sd] if not torch.equal(outs[sd][k], base[sd][k])]
        same = 'identical to first' if not bad else 'MISMATCH %s' % bad
    print('%s light=%s one_hub=%s probe_min_deg=%s ratio=%s bitmaps u/b %d/%d  user %.3f ms (light %.3f)  business %.3f ms (light %.3f)  %s' %
          (':'.join(extra), light, medium, min_deg, ratio, info['n_hub_biz'], info['n_hub_users'], res[0], lms[0], res[1], lms[1], same), flush=True)
    G.close()
