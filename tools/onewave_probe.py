import os, sys, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from new_cg_variants_b200 import PoissonStencil, Session
S = PoissonStencil(256, 256, 256, dim=3); n = S.shape[0]
b, x0 = S @ (np.ones(n)/np.sqrt(n)), np.zeros(n)
with Session(S, dinv=1/S.diagonal()) as s:
    s.load_problem(b, x0, None)
    for flag in (0, 1, 0, 1):
        s.set_option("ew_one_wave", flag)
        row = {}
        for v in ("pr", "hs", "cg", "gv", "pipe_pr"):
            best = min(s.run(v, 201, histories=(), path="stream")["loop_ms"] for _ in range(3))
            row[v] = round(1e3*best/200, 1)
        print("one_wave", flag, row, flush=True)
