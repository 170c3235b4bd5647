"""Developer tool: how the business index's bit tests spread over its 32-byte sectors (host count).

For every valid pair (u, b) of a seeded config the business side tests each id b' of N(u) against
the index.  This counts those tests exactly as the kernel makes them and, for each way of placing
the bit of (b, b') in the index, the distinct 32-byte sectors they touch and the share of tests the
hottest 32 / 64 / 96 MiB of sectors answer (an ideal cache of that size, ordered by use count; the
B200's L2 is 126 MB).  Sectors are byte address / 32 with rows of bitmap_words(n_biz) words that
start on a 256-byte boundary, as cudaMalloc places the index.  No GPU: numpy on the CPU.

Lookups (ranks: businesses by de-duplicated degree, descending, ties by id):
  id rows         row id(b), column rank(b')
  rank rows       row rank(b), column rank(b')
  symmetric       row max(rank b, rank b'), column min -- what k_score_biz_indexed reads
  transposed      row rank(b'), column rank(b)
usage: biz_sectors.py [--config C2] [--pairs N]
"""
import argparse
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SECTOR_WORDS = 8          # 32 bytes of 32-bit words
CACHE_MB = (32, 64, 96)


def bitmap_words(n):
    """blp::bitmap_words: words of a bitmap over n nodes plus the sentinel bit, multiple of 4."""
    return (((n + 1 + 31) // 32) + 3) & ~3


def tests(cfg, eu, eb, pu, pv):
    """(b, b') of every bit test the business side makes, and the business ranks."""
    nu, nb = cfg['n_users'], cfg['n_biz']
    key = np.unique(eu.astype(np.int64) * nb + eb)            # de-duplicated edges, sorted by user
    uu, bb = key // nb, key % nb
    du = np.bincount(uu, minlength=nu)
    db = np.bincount(bb, minlength=nb)
    rank = np.empty(nb, np.int64)
    rank[np.argsort(-db, kind='stable')] = np.arange(nb)
    pu, pv = pu.astype(np.int64), pv.astype(np.int64)
    ok = (pu >= 0) & (pu < nu) & (pv >= 0) & (pv < nb)
    ok[ok] = (du[pu[ok]] > 0) & (db[pv[ok]] > 0)
    pu, pv = pu[ok], pv[ok]
    d = du[pu]
    first = np.concatenate([[0], np.cumsum(du)])[pu]
    within = np.arange(int(d.sum())) - np.repeat(np.cumsum(d) - d, d)
    return np.repeat(pv, d), bb[np.repeat(first, d) + within], rank, int(ok.sum())


def sector_stats(row, col, words):
    """distinct sectors and the share of tests the hottest CACHE_MB MiB of them answer"""
    sec = (row * words + (col >> 5)) // SECTOR_WORDS
    _, counts = np.unique(sec, return_counts=True)
    hot = np.cumsum(np.sort(counts)[::-1])
    shares = [float(hot[min(hot.size, (mb << 20) // 32) - 1] / row.size) for mb in CACHE_MB]
    return counts.size, shares


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='C2')
    ap.add_argument('--pairs', type=int, default=None)
    a = ap.parse_args()
    synth = importlib.import_module('bipartite-link-prediction_b200.synth')
    cfg, eu, eb, pu, pv = synth.make_config(a.config, n_pairs=a.pairs)
    b, bp, rank, n_valid = tests(cfg, eu, eb, pu, pv)
    words = bitmap_words(cfg['n_biz'])
    rb, rbp = rank[b], rank[bp]
    print('%s: %d pairs, %d valid, %d bit tests; index %d x %d words (%.0f MB)' %
          (a.config, pu.size, n_valid, b.size, cfg['n_biz'], words, cfg['n_biz'] * words * 4 / 1e6))
    print('%-12s %19s   %s' % ('lookup', 'distinct sectors', '  '.join('%d MiB' % mb for mb in CACHE_MB)))
    for name, row, col in (('id rows', b, rbp), ('rank rows', rb, rbp),
                           ('symmetric', np.maximum(rb, rbp), np.minimum(rb, rbp)),
                           ('transposed', rbp, rb)):
        n, shares = sector_stats(row, col, words)
        print('%-12s %6.2f M (%4.0f MiB)   %s' % (name, n / 1e6, n * 32 / 2**20,
                                                  '  '.join('%.3f ' % s for s in shares)))


if __name__ == '__main__':
    main()
