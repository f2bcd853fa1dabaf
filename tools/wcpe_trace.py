import os, sys; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from dynosam_b200 import synth
from dynosam_b200.binding import Solver, default_params
from oracle import oracle as O
p = synth.make_config("C1", formulation="wcpe")
s = Solver(p); o = O.OracleProblem(p)
st = s.optimize(default_params(max_iterations=10, verbosity=1))
so = o.optimize(max_iterations=10, verbose=1)
print(st["iterations"], st["inner_iterations"], st["error_final"], so["iterations"], so["inner_iterations"], so["error_final"])
