"""Excited-state step rate on small lattices (launch-bound regime, where the CUDA-graph replay of step pairs matters):
microseconds per step for k = 1, 3 at 50^3 .. 256^3."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import wafer_b200  # noqa: E402

out = {}
for n in (50, 128, 256):
    dn = 10.24 / n
    with wafer_b200.Lattice((n,) * 3, "ThreePoint", dn=dn, dt=0.1 * dn * dn, mass=1.0) as lat:
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Boolean")
        lat.check(0)
        for k in (1, 2, 3):
            lat.push_lower()
            if k == 2:
                continue
            lat.phi_seed_from_lower(0)
            lat.check(k)
            lat.evolve(k, 200)
            lat.synchronize()
            lat.timer_begin()
            lat.evolve(k, 2000)
            ms = lat.timer_end()
            out["n%d_k%d_us_per_step" % (n, k)] = ms * 1e3 / 2000
print(json.dumps(out))
