"""Short driver for ncu: a couple of device-resident leapfrog steps of the cfg2 workload."""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from hmcmt2d_b200 import api, synthetic
ny, nz, nf = (int(a) for a in sys.argv[1:4]) if len(sys.argv) > 3 else (200, 100, 30)
nsteps = int(sys.argv[4]) if len(sys.argv) > 4 else 2
mesh, data, inv, prior = synthetic.make_problem(ny, nz, nf)
pl = api.Plan(mesh, data, inv, prior)
m = synthetic.stress_model(inv)
pl.set_state(m, np.clip(np.random.default_rng(0).standard_normal(len(m)), -2.5, 2.5), m)
pl.leapfrog_steps_device(prior.dt, nsteps)
pl.sync()
print("done", pl.info(10), "launches")
