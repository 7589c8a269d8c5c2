"""Parity of the paths the small-lattice suite does not reach, against the CPU oracle.

* the time-tiled sweep with the work distribution of the benchmark (1024^3: several x chunks, several rounds of whole
  tile columns handed out through the atomic counter, a statically cut tail), checked site by site against light-cone
  boxes of the numpy restatement, and at moderate sizes whose plans have the same structures, against the whole oracle;
* state cached on a context across calls: the CUDA graphs of excited-state steps, the h field of the time-tiled sweep,
  the check sums fused into the last sweep of an evolve;
* the A/B switch read from the environment (WAFER_T1_HFIELD, one worker process per setting), which must not change a
  single bit.

Bars as in test_gpu_parity.py: bit for bit where nothing is reduced, 1e-12 relative for sums and excited-state steps.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import np_restatement as npr

gpu = pytest.mark.gpu

SUM_TOL = 1e-12
TY, TZ = 30, 60  # output tile of sweep_tb.cuh


@pytest.fixture(scope="module")
def wb():
    import wafer_b200
    return wafer_b200


def _l2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _work_random(g, rng, scale=1.0):
    phi = np.zeros(g.padded_shape)
    npr.work(phi, g.ext)[...] = rng.normal(size=g.work_shape) * scale
    return phi


def _plan_structure(plan, slots):
    """(x chunks of the bulk, whole rounds of the bulk, tail segment lengths) of a wafer_b200.tb2_plan array"""
    bulk, tail = plan[plan[:, 0] < 0], plan[plan[:, 0] >= 0]
    assert len(bulk) % slots == 0
    return len({(a, z) for a, z in bulk[:, 3:5]}), len(bulk) // slots, tail[:, 4] - tail[:, 3]


# ---------------------------------------------------------------------------------------------- plan structures, full oracle
# (nx, ny, nz), x chunks, bulk rounds on 148 SMs.  (40, 512, 512): 14 tail columns of 40 planes are less than 6 planes per
# CTA, so only some CTAs get a tail share (before that was fixed, every CTA got one, of 2 or 4 planes).
PLAN_SHAPES = [((40, 512, 512), 1, 1), ((600, 390, 720), 2, 2), ((160, 600, 1080), 3, 7)]


@gpu
@pytest.mark.parametrize("shape,chunks,rounds", PLAN_SHAPES)
def test_time_tiled_sweep_with_chunks_rounds_and_tail(wb, oracle, shape, chunks, rounds):
    """Three evolves on one context (the schedule is cached and its counters re-arm themselves between launches):
    3 steps before the h field exists = one time-tiled launch that reads V and one one-step step; 7 steps = the h field,
    three time-tiled launches that read it and one one-step tail step; then 6 more."""
    rng = np.random.default_rng(97)
    g = oracle.make_grid(*shape, ext=1, dn=0.05, dt=6.25e-4, mass=1.0)
    v = rng.normal(size=g.padded_shape) * 3.0
    phi = _work_random(g, rng)
    a, b = oracle.build_ab(v, g.dt)
    with wb.Lattice(shape, dn=g.dn, dt=g.dt, mass=g.mass) as lat:
        slots = lat.device_info()["sm_count"]  # one CTA per SM (sweep_tb.cuh CTAS_PER_SM)
        nc, nr, tail = _plan_structure(wb.tb2_plan(shape[1], shape[2], 0, shape[0], slots), slots)
        if slots == 148:
            assert (nc, nr) == (chunks, rounds)
        assert nc >= 1 and nr >= 1 and len(tail) > 0 and tail.min() >= 6, (nc, nr, tail)
        lat.set_potential(v)
        lat.set_phi(phi)
        lat.evolve(0, 3)
        got3 = lat.get_phi()
        lat.evolve(0, 7)
        got7 = lat.get_phi()
        lat.evolve(0, 6)
        got13 = lat.get_phi()
    oracle.evolve(g, phi, a, b, 3)
    assert np.array_equal(got3, phi)
    oracle.evolve(g, phi, a, b, 7)
    assert np.array_equal(got7, phi)
    oracle.evolve(g, phi, a, b, 6)
    assert np.array_equal(got13, phi)


# ---------------------------------------------------------------------------------------------- 1024^3, light cones
def light_cone_values(psi0, v, sites, steps, dn, dt, mass):
    """psi after `steps` ThreePoint sweeps at `sites` (padded indices), from psi0 and V alone: a site depends only on
    the sites within distance `steps`, so sweeping the box of half-width steps + 1 around it (clipped to the padded
    lattice; its faces stay frozen like the lattice's ring) gives the centre exactly."""
    h = steps + 1
    out = np.empty(len(sites))
    for i, (x, y, z) in enumerate(sites):
        lo = [max(c - h, 0) for c in (x, y, z)]
        hi = [min(c + h + 1, n) for c, n in zip((x, y, z), psi0.shape)]
        box = np.s_[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]]
        p = np.array(psi0[box])
        a, b = npr.build_ab(np.array(v[box]), dt)
        for _ in range(steps):
            p = npr.sweep(p, a, b, 1, dn, dt, mass)
        out[i] = p[x - lo[0], y - lo[1], z - lo[2]]
    return out


def sample_sites(n, plan, seed, n_seam=3000, n_random=2000):
    """padded indices of (seams, faces, random) sites of an n^3 lattice.  Seams: tile edges (y near multiples of TY,
    z near multiples of TZ) on the first and last two planes of every bulk chunk and every tail segment; for a tail
    segment, at the edges of its own tile."""
    rng = np.random.default_rng(seed)
    ys = sorted({y for m in range(1, -(-n // TY)) for y in (m * TY - 1, m * TY, m * TY + 1)} - {n})
    zs = sorted({z for m in range(1, -(-n // TZ)) for z in (m * TZ - 2, m * TZ - 1, m * TZ, m * TZ + 1)} - {n})
    ys = [y for y in ys if y < n]
    zs = [z for z in zs if z < n]
    edge = lambda a, z: {a, a + 1, z - 2, z - 1} & set(range(a, z))
    bulk, tail = plan[plan[:, 0] < 0], plan[plan[:, 0] >= 0]
    bulk_planes = sorted({x for a, z in {(a, z) for a, z in bulk[:, 3:5]} for x in edge(a, z)})
    seams = set()
    for _ in range(n_seam // 2):
        seams.add((rng.choice(bulk_planes), rng.choice(ys), rng.choice(zs)))
    for _, y0, z0, xa, xz in tail[rng.permutation(len(tail))[:n_seam // 8]]:
        for x in edge(xa, xz):
            y = rng.choice([c for c in (y0 - 1, y0, y0 + 1, y0 + TY - 1, y0 + TY) if 0 <= c < n])
            z = rng.choice([c for c in (z0 - 2, z0 - 1, z0, z0 + 1, z0 + TZ - 1, z0 + TZ) if 0 <= c < n])
            seams.add((x, y, z))
    ends = (0, 1, n // 2, n - 2, n - 1)
    faces = {(x, y, z) for x in ends for y in ends for z in ends if {x, y, z} & {0, n - 1}}
    for ax in range(3):
        for side in (0, n - 1):
            for _ in range(50):
                c = list(rng.integers(0, n, 3))
                c[ax] = side
                faces.add(tuple(c))
    rand = {tuple(c) for c in rng.integers(0, n, (n_random, 3))}
    pad = lambda s: np.array(sorted(s), dtype=np.int64).reshape(-1, 3) + 1
    return pad(seams), pad(faces), pad(rand)


def test_light_cone_sampler_compares_values(oracle):
    """CPU check of the sampler itself: exact against the whole oracle, and one ulp in one input is seen."""
    n, steps = 64, 7
    rng = np.random.default_rng(5)
    g = oracle.make_grid(n, n, n, ext=1, dn=0.05, dt=6.25e-4, mass=1.0)
    v = rng.normal(size=g.padded_shape) * 3.0
    psi0 = _work_random(g, rng)
    a, b = oracle.build_ab(v, g.dt)
    ref = psi0.copy()
    oracle.evolve(g, ref, a, b, steps)
    plan = np.array([[-1, 0, 0, 0, 32], [-1, 30, 0, 32, 64], [0, 0, 60, 32, 40], [1, 30, 60, 40, 64]], dtype=np.int32)
    sites = np.concatenate(sample_sites(n, plan, 1, n_seam=200, n_random=100))
    got = light_cone_values(psi0, v, sites, steps, g.dn, g.dt, g.mass)
    assert np.array_equal(got, ref[tuple(sites.T)])
    # one ulp more in one input of a box: the boxes follow the oracle bit for bit, and the comparison sees the change
    # wherever it reaches the output (after 7 steps a single ulp may also round away)
    seen = 0
    for i in range(0, len(sites), 37):
        x, y, z = sites[i]
        bumped = psi0.copy()
        bumped[x, y, z] = np.nextafter(bumped[x, y, z], np.inf)
        ref2 = bumped.copy()
        oracle.evolve(g, ref2, a, b, steps)
        mine = light_cone_values(bumped, v, sites[i:i + 1], steps, g.dn, g.dt, g.mass)[0]
        assert mine == ref2[x, y, z]
        seen += mine != got[i]
    assert seen >= 3, seen


def _mem_available():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


@gpu
def test_benchmark_workload_1024_cubed_site_by_site(wb):
    """Workload C4 (bench.py): 1024^3 Poschl-Teller, Boolean start, 7 steps = three time-tiled launches (4 x chunks,
    17 rounds through the counter, a static tail; counter re-armed twice; h field) + one one-step tail step.  Sampled
    sites against light-cone boxes; the whole field against the register-queue and the TMA one-step sweeps."""
    n, steps = 1024, 7
    field = (n + 2) ** 3 * 8
    if _mem_available() < 40e9:  # three host copies of the field + boxes: about 30 GB (estimate)
        pytest.skip("needs about 40 GB of available host memory for three 8.6 GB copies of the 1024^3 field")
    dn = 10.24 / n
    dt, mass = 0.3 * dn * dn, 1.0
    try:
        lat = wb.Lattice((n, n, n), dn=dn, dt=dt, mass=mass)
    except wb.WaferError as e:
        pytest.skip("the device cannot hold the 1024^3 fields: %s" % e)
    out = None
    try:
        info = lat.device_info()
        if info["mem_bytes"] < 5 * field:
            pytest.skip("the device cannot hold the 1024^3 fields (%d bytes)" % info["mem_bytes"])
        assert lat.sweep_variant.startswith("tb2")
        lat.generate_potential("PoschlTeller")
        lat.set_initial_conditions("Boolean")
        psi0 = lat.get_phi()
        v = lat.get_potential()  # device libm (cosh): not a host formula
        lat.evolve(0, steps)
        out = wb.pinned_empty(lat.padded_shape)
        lat.get_phi(out)
        tiled = lat.phi_checksum()
        plan = wb.tb2_plan(n, n, 0, n, slots=info["sm_count"])
        lat.close()
        seams, faces, rand = sample_sites(n, plan, 2024)
        for name, sites in (("seams", seams), ("faces", faces), ("random", rand)):
            want = light_cone_values(psi0, v, sites, steps, dn, dt, mass)
            got = out[tuple(sites.T)]
            bad = np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))
            assert len(bad) == 0, (name, len(sites), [tuple(s) for s in sites[bad[:5]]])
        print("\n1024^3 light cones: %d seam, %d face, %d random sites bit-exact" % (len(seams), len(faces), len(rand)))
        del psi0, v
        sums = {"tb2": tiled}
        for flags in (4, 12):  # register-queue one-step sweep; TMA one-step sweep only
            with wb.Lattice((n, n, n), dn=dn, dt=dt, mass=mass, flags=flags) as other:
                other.generate_potential("PoschlTeller")
                other.set_initial_conditions("Boolean")
                other.evolve(0, steps)
                sums[other.sweep_variant] = other.phi_checksum()
        print("1024^3 phi_checksum after %d steps: %s" % (steps, sums))
        assert len(set(sums.values())) == 1, sums
    finally:
        lat.close()
        if out is not None:
            wb.pinned_free(out)


# ---------------------------------------------------------------------------------------------- cached state: graphs
def _excited_case(oracle, nlow, seed, shape=(18, 16, 22)):
    rng = np.random.default_rng(seed)
    g = oracle.make_grid(*shape, ext=1, dn=0.1, dt=2e-3, mass=1.0)
    v = oracle.potential(g, "Harmonic")
    lowers = []
    for _ in range(nlow):
        q = npr.orthogonalise(_work_random(g, rng), lowers)
        lowers.append(np.ascontiguousarray(q / np.sqrt((q * q).sum())))
    return g, v, lowers, _work_random(g, rng)


def _stepwise(wb, g, v, lowers, phi, wnum, pre, steps, flags):
    """`pre` steps, then `steps` steps, one evolve(wnum, 1) call each: never a graph"""
    with wb.Lattice(g.work_shape, dn=g.dn, dt=g.dt, mass=g.mass, flags=flags) as lat:
        lat.set_potential(v)
        for q in lowers:
            lat.push_lower(q)
        lat.set_phi(phi)
        for _ in range(pre + steps):
            lat.evolve(wnum, 1)
        return lat.get_phi()


def _oracle_excited(oracle, g, v, lowers, phi, steps):
    a, b = oracle.build_ab(v, g.dt)
    ref = phi.copy()
    oracle.set_sum_mode(1)
    try:
        oracle.evolve(g, ref, a, b, steps, lowers=lowers)
    finally:
        oracle.set_sum_mode(0)
    return ref


@gpu
@pytest.mark.parametrize("flags", [0, 4])
@pytest.mark.parametrize("pre", [0, 1])  # an extra single step first: the graph of the other buffer parity
@pytest.mark.parametrize("steps", [8, 9])
@pytest.mark.parametrize("wnum", [1, 4])
def test_graph_replay_equals_single_steps(wb, oracle, wnum, steps, pre, flags):
    g, v, lowers, phi = _excited_case(oracle, wnum, 3 + wnum)
    with wb.Lattice(g.work_shape, dn=g.dn, dt=g.dt, mass=g.mass, flags=flags) as lat:
        lat.set_potential(v)
        for q in lowers:
            lat.push_lower(q)
        lat.set_phi(phi)
        if pre:
            lat.evolve(wnum, 1)
        lat.evolve(wnum, steps)
        got = lat.get_phi()
    assert np.array_equal(got, _stepwise(wb, g, v, lowers, phi, wnum, pre, steps, flags))
    assert _l2(got, _oracle_excited(oracle, g, v, lowers, phi, pre + steps)) < 1e-12


@gpu
@pytest.mark.parametrize("flags", [0, 4])
def test_graph_cache_follows_the_store_and_the_potential(wb, oracle, flags):
    """A captured graph holds the addresses of the stored states: it must not outlive them, and a different wnum or a new
    potential must be seen by the next replay."""
    g, v, lowers, phi = _excited_case(oracle, 2, 11)
    _, _, others, _ = _excited_case(oracle, 3, 12)
    v2 = np.ascontiguousarray(v * 0.5 + 1.0)
    with wb.Lattice(g.work_shape, dn=g.dn, dt=g.dt, mass=g.mass, flags=flags) as lat:
        lat.set_potential(v)
        for q in lowers:
            lat.push_lower(q)

        def run(wnum, store, pot):
            lat.set_phi(phi)
            lat.evolve(wnum, 8)
            got = lat.get_phi()
            assert np.array_equal(got, _stepwise(wb, g, pot, store, phi, wnum, 0, 8, flags)), (wnum, len(store))
            assert _l2(got, _oracle_excited(oracle, g, pot, store[:wnum], phi, 8)) < 1e-12

        run(2, lowers, v)                     # captures the graph of (wnum 2, this parity)
        lat.clear_lowers()                    # frees the states the graph read
        for q in others[:2]:
            lat.push_lower(q)
        run(2, others[:2], v)
        lat.push_lower(others[2])
        run(3, others, v)
        run(2, others, v)
        lat.set_potential(v2)
        run(2, others, v2)
        run(3, others, v2)


# ---------------------------------------------------------------------------------------------- cached state: h field
@gpu
@pytest.mark.parametrize("how", ["set", "generate"])
def test_h_field_is_rebuilt_when_the_potential_changes(wb, oracle, how):
    """evolve(0, >= 4) builds h = (dt V)/2 once; a new potential must drop it (evolve(0, 2) then reads V, and
    evolve(0, 4) builds h again from the new V)."""
    shape = (40, 33, 70)
    rng = np.random.default_rng(13)
    g = oracle.make_grid(*shape, ext=1, dn=0.05, dt=6.25e-4, mass=1.0)
    phi = _work_random(g, rng)
    with wb.Lattice(shape, dn=g.dn, dt=g.dt, mass=g.mass) as lat:
        if how == "set":
            lat.set_potential(rng.normal(size=g.padded_shape) * 3.0)
        else:
            lat.generate_potential("Harmonic")
        v1 = lat.get_potential()
        lat.set_phi(phi)
        lat.evolve(0, 4)
        got = lat.get_phi()
        ref = phi.copy()
        oracle.evolve(g, ref, *oracle.build_ab(v1, g.dt), 4)
        assert np.array_equal(got, ref)
        if how == "set":
            lat.set_potential(rng.normal(size=g.padded_shape) * 3.0)
        else:
            lat.generate_potential("QuadWell")
        v2 = lat.get_potential()
        assert not np.array_equal(npr.work(v1, 1), npr.work(v2, 1))
        a2, b2 = oracle.build_ab(v2, g.dt)
        for steps in (2, 4):
            lat.set_phi(phi)
            lat.evolve(0, steps)
            got = lat.get_phi()
            ref = phi.copy()
            oracle.evolve(g, ref, a2, b2, steps)
            assert np.array_equal(got, ref), steps


# ---------------------------------------------------------------------------------------------- cached state: fused check sums
@gpu
@pytest.mark.parametrize("change", ["pot_sub_scalar", "pot_sub_array", "set_phi", "normalise", "phi_from_lower",
                                    "phi_seed_from_lower"])
def test_fused_check_sums_are_dropped_when_their_inputs_change(wb, oracle, change):
    """evolve(0, >= 64) leaves sum psi^2, sum psi^2 pot_sub and sum psi^2 r2 of its last sweep for the next check;
    after any call that changes psi or pot_sub, observables and check must describe the new state."""
    shape = (22, 35, 61)
    rng = np.random.default_rng(29)
    g = oracle.make_grid(*shape, ext=1, dn=0.1, dt=6.25e-4, mass=1.0)
    v = rng.normal(size=g.padded_shape) * 0.3
    phi = _work_random(g, rng)
    q = _work_random(g, rng)
    ps = None
    with wb.Lattice(shape, dn=g.dn, dt=g.dt, mass=g.mass) as lat:
        lat.set_potential(v)
        lat.push_lower(q)
        lat.set_phi(phi)
        lat.evolve(0, 64)
        state = lat.get_phi()
        if change == "pot_sub_scalar":
            ps = 2.5
            lat.set_pot_sub(ps)
        elif change == "pot_sub_array":
            ps = rng.uniform(0.5, 2.0, size=shape)
            lat.set_pot_sub(ps)
        elif change == "set_phi":
            state = _work_random(g, rng)
            lat.set_phi(state)
        elif change == "normalise":
            lat.normalise_wavefunction(3.7)
            oracle.normalise(state, 3.7)
        elif change == "phi_from_lower":
            lat.phi_from_lower(0)
            state = q.copy()
        else:
            lat.phi_seed_from_lower(0)
            state = oracle.seed_from_state(g, q)
        assert np.array_equal(lat.get_phi(), state)
        oracle.set_sum_mode(1)
        try:
            want = oracle.observables(g, state, v, ps)
        finally:
            oracle.set_sum_mode(0)
        scale = max(abs(want["energy"]), want["norm2"], abs(want["r2"]))
        for got in (lat.compute_observables(), lat.check(0)):
            for key in want:
                assert abs(got[key] - want[key]) <= SUM_TOL * scale, (key, got[key], want[key])


# ---------------------------------------------------------------------------------------------- environment switch
ENV_VARIANTS = [{}, {"WAFER_T1_HFIELD": "1"}]
ENV_KEYS = sorted({k for e in ENV_VARIANTS for k in e})


def worker():
    """Fixed workloads, generated on the device; prints {name: phi_checksum} as one JSON line."""
    import wafer_b200 as wb
    sums = {}
    with wb.Lattice((160, 600, 1080), dn=0.01, dt=3e-5) as lat:  # 3 x chunks, 7 rounds, a tail
        lat.generate_potential("PoschlTeller")
        lat.set_initial_conditions("Boolean")
        lat.evolve(0, 7)
        sums["tb2_7"] = lat.phi_checksum()
    with wb.Lattice((64, 90, 130), "FivePoint", dn=0.05, dt=6.25e-4) as lat:
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Coulomb")
        lat.evolve(0, 3)
        sums["five_point_3"] = lat.phi_checksum()
    with wb.Lattice((40, 50, 66), dn=0.1, dt=2e-3) as lat:
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Boolean")
        lat.evolve(0, 4)
        lat.normalise_wavefunction(lat.get_norm_squared())
        lat.push_lower()
        lat.phi_seed_from_lower(0)
        lat.orthogonalise_wavefunction(1)
        lat.normalise_wavefunction(lat.get_norm_squared())
        lat.push_lower()
        lat.phi_seed_from_lower(1)
        lat.evolve(2, 9)
        sums["excited_2_9"] = lat.phi_checksum()
    print(json.dumps({k: list(v) for k, v in sums.items()}))


@gpu
def test_environment_switches_give_identical_results():
    """The switch is read once per process: one worker per setting, each must print the default's checksums."""
    here = os.path.abspath(__file__)
    results = []
    for extra in ENV_VARIANTS:
        env = {k: v for k, v in os.environ.items() if k not in ENV_KEYS}
        env.update(extra)
        r = subprocess.run([sys.executable, here, "--worker"], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (extra, r.stdout[-2000:], r.stderr[-2000:])
        results.append((extra, json.loads(r.stdout.strip().splitlines()[-1])))
    base = results[0][1]
    assert set(base) == {"tb2_7", "five_point_3", "excited_2_9"}
    for extra, sums in results[1:]:
        assert sums == base, extra


if __name__ == "__main__" and sys.argv[1:] == ["--worker"]:
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    worker()
