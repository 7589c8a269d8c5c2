"""Excited-state step rate at 512^3 for k = 3, 4 stored states (the modes of the one-step sweep that prefetch one of the
stored states)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import wafer_b200  # noqa: E402

n = 512
dn = 10.24 / n
out = {"lib": os.path.basename(os.environ.get("WAFER_B200_LIB", "default"))}
with wafer_b200.Lattice((n,) * 3, "ThreePoint", dn=dn, dt=0.1 * dn * dn, mass=1.0) as lat:
    lat.generate_potential("Harmonic")
    lat.set_initial_conditions("Boolean")
    lat.check(0)
    for k in (1, 2, 3, 4):
        lat.push_lower()
        if k < 3:
            continue
        lat.phi_seed_from_lower(0)
        lat.check(k)
        lat.evolve(k, 10)
        lat.synchronize()
        lat.timer_begin()
        lat.evolve(k, 40)
        ms = lat.timer_end()
        out["k%d_glups" % k] = n ** 3 * 40 / ms / 1e6
print(json.dumps(out))
