#!/usr/bin/env python
"""apply_r.lua's main() through the B200 library: python tools/apply_r_main.py [--G x.net --R y.net --R_fixer z.net] --writeTo r_results"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from __graft_entry__ import load_package

ap = argparse.ArgumentParser()
ap.add_argument("--G"); ap.add_argument("--R"); ap.add_argument("--R_fixer")
ap.add_argument("--writeTo", default="r_results"); ap.add_argument("--seed", type=int, default=1)
ap.add_argument("--gpu", type=int, default=0); ap.add_argument("--images", type=int, default=10000)
ap.add_argument("--refine", type=int, default=0, metavar="ITERS",
                help="also refine the fixer's vectors by ITERS Adam steps through G and write fixed_refined.jpg / anomalies_refined.jpg")
a = ap.parse_args()
pkg = load_package()
ctx = pkg.Context(a.gpu)
out = pkg.apply_r.main(G=a.G, R=a.R, R_fixer=a.R_fixer, writeTo=a.writeTo, seed=a.seed, nbImages=a.images, ctx=ctx, refine=a.refine)
print("\n".join(out["files"]))
