import os, sys; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from dynosam_b200 import synth
from dynosam_b200.binding import Solver
from oracle import oracle as O
p = synth.make_problem(n_frames=400, n_objects=4, n_static=4000, n_dynamic=2000, formulation="hybrid", seed=13, object_span=(120, 200))
s = Solver(p); o = O.OracleProblem(p)
print(s.info())
lam=1e-4
d = s.solve(lam); rc, do = o.schur_solve(lam)
H,g = o.dense_normal() if p.n_pose*6+p.n_point*3 < 30000 else (None,None)
print("step rel err vs oracle", np.linalg.norm(d-do)/np.linalg.norm(do))
if H is not None:
    dd = np.linalg.solve(H+lam*np.eye(H.shape[0]), g)
    print("gpu vs dense", np.linalg.norm(d-dd)/np.linalg.norm(dd), " oracle vs dense", np.linalg.norm(do-dd)/np.linalg.norm(dd))
st = s.optimize(max_iterations=6); so = o.optimize(max_iterations=6)
print(st["error_final"], so["error_final"], abs(st["error_final"]-so["error_final"])/so["error_final"], st["iterations"], so["iterations"])
