"""Lattice statistics that decide K3's design (run on the CPU with the analysis build of the oracle).

For the synthetic workloads of bench.py: how many distinct right ids a lattice row has, how many distinct left
ids the candidates of a position have (the gain of de-duplicating connection-cost lookups), and how many
(candidate, predecessor) pairs survive an exact lower-bound pruning.  Writes a markdown table to stdout.

    python tools/lattice_stats.py [--dict synth-unidic] [--n 20000] [--fixed-len 0]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vibrato_b200 import synth  # noqa: E402
import oracle.vibrato_oracle as vo  # noqa: E402

NAMES = ["calls", "pairs", "distinct_right", "surv_colmin", "surv_both", "surv_sorted", "positions", "cands",
         "distinct_left", "distinct_pairs", "surv_natural", "surv_natural_both", "surv_heur",
         "first_static", "first_b4", "argmin_b4", "last_b4"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dict", default="synth-unidic")
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--fixed-len", type=int, default=0)
    a = ap.parse_args()
    so = os.path.join(ROOT, "tools", "_build", "liboracle_ana.so")
    src = os.path.join(ROOT, "oracle", "vibrato_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-fPIC", "-std=gnu11", "-pthread", "-DVO_ANALYSIS",
                               "-shared", "-o", so, src])
    vo._SO = so
    L = vo.lib()
    sd = synth.make_dictionary(a.dict)
    kw = dict(fixed_len=a.fixed_len) if a.fixed_len else {}
    utf8, off = synth.make_corpus(sd, a.n, seed=20260923 + 2, **kw)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    L.vo_ana_prepare.argtypes = [C.c_void_p]
    L.vo_ana_prepare(od._h if hasattr(od, "_h") else od.handle)
    od.tokenize_batch(utf8, off, n_threads=1, want_tokens=False)
    ana = (C.c_uint64 * len(NAMES)).in_dll(L, "vo_ana")
    v = dict(zip(NAMES, [int(x) for x in ana]))
    print(f"| {a.dict}, {a.n} sentences" + (f" x {a.fixed_len} chars" if a.fixed_len else "") + " | value |")
    print("|---|---:|")
    print(f"| connection-cost lookups (pairs) | {v['pairs']} |")
    print(f"| predecessors per search (K) | {v['pairs'] / v['calls']:.2f} |")
    print(f"| distinct right ids / predecessors | {v['distinct_right'] / v['pairs']:.3f} |")
    print(f"| candidates per visited position | {v['cands'] / v['positions']:.2f} |")
    print(f"| distinct left ids / candidates | {v['distinct_left'] / v['cands']:.3f} |")
    print(f"| distinct (left, right) pairs / pairs | {v['distinct_pairs'] / v['pairs']:.3f} |")
    print(f"| pairs surviving bound min_r M[l][r] after the cheapest predecessor | {v['surv_colmin'] / v['pairs']:.3f} |")
    print(f"| ... with max(min_r M[l][.], min_l M[.][r]) | {v['surv_both'] / v['pairs']:.3f} |")
    print(f"| ... row order with a running best, bound min_r M[l][r] | {v['surv_natural'] / v['pairs']:.3f} |")
    print(f"| ... row order, running best, both bounds | {v['surv_natural_both'] / v['pairs']:.3f} |")
    print(f"| ... cheapest of the first 8 predecessors first, then row order with a running best | {v['surv_heur'] / v['pairs']:.3f} |")
    print(f"| GPU schedule: row's first predecessor alone, others against its total | {v['first_static'] / v['pairs']:.3f} |")
    print(f"| GPU schedule: first alone, then batches of 4 (bound = best before the batch) | {v['first_b4'] / v['pairs']:.3f} |")
    print(f"| GPU schedule: cheapest alone, then all in row order in batches of 4 | {v['argmin_b4'] / v['pairs']:.3f} |")
    print(f"| GPU schedule: row's last predecessor alone, then batches of 4 | {v['last_b4'] / v['pairs']:.3f} |")
    print(f"| ... ascending predecessor cost, running best, both bounds | {v['surv_sorted'] / v['pairs']:.3f} |")


if __name__ == "__main__":
    main()
