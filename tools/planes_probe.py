import os, sys, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from new_cg_variants_b200 import PoissonStencil, Session
for shape in ((256,256,32),(256,256,16),(256,256,64),(64,64,64)):
    S = PoissonStencil(*shape, dim=3); n = S.shape[0]
    b, x0 = S @ (np.ones(n)/np.sqrt(n)), np.zeros(n)
    with Session(S, dinv=1/S.diagonal()) as s:
        s.load_problem(b, x0, None)
        for mp in (2, 4, 6, 8, 12, 16):
            s.set_option("tma_min_planes", mp)
            row = {}
            for v in ("pr", "pipe_pr"):
                best = min(s.run(v, 201, histories=(), path="stream")["loop_ms"] for _ in range(3))
                row[v] = round(1e3*best/200, 1)
            print(shape, "min_planes", mp, row, flush=True)
