"""init_symmetry (config.rs:186-197, 625, 691-728; grid.rs:137-139) and the seeded Gaussian initial condition
(config.rs:636-642), made on the device by wafer_symmetrise / wafer_generate_gaussian.

Definitions (DESIGN.md "Initial state"):
* mirror: with n the work size of the mirrored axis (z for AboutZ / AntisymAboutZ, y for AboutY / AntisymAboutY),
  psi[.., n-1-t] = s psi[.., t] for t < n/2, s = +1 / -1; for odd n the middle index is kept (s = +1) or set to +0.
* Gaussian: Philox4x32-10 with key (lo32(seed), hi32(seed)) and counter (lo32(s), hi32(s), 0, 0) at the global work
  index s = (i*ny + j)*nz + k; u1 = ((r0>>5) 2^26 + (r1>>6) + 1) 2^-53, u2 = ((r2>>5) 2^26 + (r3>>6)) 2^-53;
  value = sig * (sqrt(-2 log u1) * cos(2 pi u2)).

The mirror is a copy and a sign flip, so it is compared bit for bit; the Gaussian goes through the device's log and cos,
which may differ from numpy's by an ulp or two.
"""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import np_restatement as npr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "wafer_b200", "wafer-b200")
DEFAULT = os.path.join(ROOT, "tests", "golden", "wafer_default.yaml")

gpu = pytest.mark.gpu

SUM_TOL = 1e-12
CD = {1: "ThreePoint", 2: "FivePoint", 3: "SevenPoint"}
SYMMETRIES = ["NotConstrained", "AboutZ", "AntisymAboutZ", "AboutY", "AntisymAboutY"]
FLAG_NO_FUSED_CHECK = 0x10
ROW = re.compile(r"\s+│\s+[0-9.]+ │")


@pytest.fixture(scope="module")
def wb():
    import wafer_b200
    return wafer_b200


@pytest.fixture(scope="module")
def binary():
    if not os.path.exists(BIN):
        import __graft_entry__
        __graft_entry__.build()
    return BIN


# ---------------------------------------------------------------------------------------------- numpy restatements
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Random123 constants) on uint64 arrays holding 32-bit words; returns the four output words"""
    c = [np.asarray(x, dtype=np.uint64) for x in ctr]
    k0, k1 = (np.asarray(x, dtype=np.uint64) for x in key)
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
            k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _M32]
    return c


def np_gaussian(size, ext, sig, seed):
    """the padded array wafer_generate_gaussian makes (ring 0)"""
    s = np.arange(int(np.prod(size)), dtype=np.uint64)
    zero = np.zeros_like(s)
    seed = np.uint64(seed)
    r = philox4x32_10((s & _M32, s >> np.uint64(32), zero, zero), (seed & _M32, seed >> np.uint64(32)))
    u1 = ((r[0] >> np.uint64(5)).astype(np.float64) * 67108864.0 + (r[1] >> np.uint64(6)).astype(np.float64) + 1.0) * 2.0 ** -53
    u2 = ((r[2] >> np.uint64(5)).astype(np.float64) * 67108864.0 + (r[3] >> np.uint64(6)).astype(np.float64)) * 2.0 ** -53
    val = sig * (np.sqrt(-2.0 * np.log(u1)) * np.cos(6.283185307179586 * u2))
    out = np.zeros(tuple(n + 2 * ext for n in size))
    npr.work(out, ext)[...] = val.reshape(size)
    return out


def np_symmetrise(phi, ext, kind):
    """the mirror of wafer_symmetrise on a padded array (kind: SymmetryConstraint index)"""
    kind = SYMMETRIES.index(kind) if isinstance(kind, str) else kind
    out = phi.copy()
    if kind == 0:
        return out
    w = npr.work(out, ext)
    axis = 2 if kind in (1, 2) else 1
    sign = -1.0 if kind in (2, 4) else 1.0
    n = w.shape[axis]
    wm = np.moveaxis(w, axis, 0)  # a view: writes go to `out`
    for t in range(n // 2):
        wm[n - 1 - t] = sign * wm[t]
    if n % 2 and sign < 0:
        wm[n // 2] = 0.0
    return out


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _ring_is_zero(a, ext):
    inner = np.zeros(a.shape, dtype=bool)
    npr.work(inner, ext)[...] = True
    return not _bits(a)[~inner].any()  # +0.0 bits, not only == 0


def _random_phi(shape, ext, seed):
    rng = np.random.default_rng(seed)
    phi = np.zeros(tuple(n + 2 * ext for n in shape))
    npr.work(phi, ext)[...] = rng.normal(size=shape)
    return phi


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_numpy_philox_matches_known_answers(ctr, key, want):
    """Random123 kat_vectors for philox4x32_10"""
    assert tuple(int(x) for x in philox4x32_10(ctr, key)) == want


def test_numpy_mirror_definition():
    phi = _random_phi((3, 5, 7), 1, 0)
    for kind in range(1, 5):
        once = np_symmetrise(phi, 1, kind)
        assert np.array_equal(_bits(np_symmetrise(once, 1, kind)), _bits(once))
        w = npr.work(once, 1)
        ax = 2 if kind in (1, 2) else 1
        s = -1.0 if kind in (2, 4) else 1.0
        assert np.array_equal(np.flip(w, ax), s * w)
    w = npr.work(np_symmetrise(phi, 1, 2), 1)
    assert np.array_equal(w[..., :3], npr.work(phi, 1)[..., :3]) and not w[..., 3].any()


def _check(binary, text, tmp_path, *extra):
    cfg = tmp_path / "wafer.yaml"
    cfg.write_text(text)
    return subprocess.run([binary, "-c", str(cfg), "--check-config", *extra], capture_output=True, text=True)


def test_check_config_accepts_every_symmetry(binary, tmp_path):
    base = open(DEFAULT).read()
    for name in SYMMETRIES:
        r = _check(binary, base.replace("init_symmetry: NotConstrained", "init_symmetry: " + name), tmp_path)
        assert r.returncode == 0, (name, r.stderr)
        assert json.loads(r.stdout)["init_symmetry"] == name
    r = _check(binary, base.replace("init_symmetry: NotConstrained", "init_symmetry: AntisymAboutX"), tmp_path)
    assert r.returncode == 1 and "unknown variant" in r.stderr


def test_check_config_refuses_antisymmetry_about_a_single_site(binary, tmp_path):
    """the antisymmetric state about an axis of work size 1 is zero everywhere"""
    base = open(DEFAULT).read()
    r = _check(binary, base.replace("z: 50", "z: 1").replace("NotConstrained", "AntisymAboutZ"), tmp_path)
    assert r.returncode == 1 and "AntisymAboutZ" in r.stderr and "along z" in r.stderr
    r = _check(binary, base.replace("y: 50", "y: 1").replace("NotConstrained", "AntisymAboutY"), tmp_path)
    assert r.returncode == 1 and "AntisymAboutY" in r.stderr and "along y" in r.stderr
    for text in (base.replace("z: 50", "z: 1").replace("NotConstrained", "AboutZ"),
                 base.replace("y: 50", "y: 1").replace("NotConstrained", "AntisymAboutZ"),
                 base.replace("z: 50", "z: 1").replace("NotConstrained", "AntisymAboutY")):
        r = _check(binary, text, tmp_path)
        assert r.returncode == 0, r.stderr


def test_seed_option_is_parsed(binary, tmp_path):
    base = open(DEFAULT).read()
    assert json.loads(_check(binary, base, tmp_path).stdout)["seed"] == 0  # the documented default
    for seed in ("12345", str(2 ** 64 - 1)):
        r = _check(binary, base, tmp_path, "--seed", seed)
        assert r.returncode == 0 and json.loads(r.stdout)["seed"] == int(seed), r.stderr
    for bad in ("-1", "abc", "12x", str(2 ** 64), ""):
        r = _check(binary, base, tmp_path, "--seed", bad)
        assert r.returncode == 2 and "--seed" in r.stderr, bad
    assert "--seed" in subprocess.run([binary, "--help"], capture_output=True, text=True).stdout


# ---------------------------------------------------------------------------------------------- GPU: the mirror
MIRROR_SHAPES = [(20, 33, 40), (17, 16, 31), (9, 1, 70), (9, 40, 1)]


@gpu
@pytest.mark.parametrize("shape", MIRROR_SHAPES)
@pytest.mark.parametrize("ext", [1, 2, 3])
@pytest.mark.parametrize("kind", SYMMETRIES[1:])
def test_symmetrise_matches_numpy_mirror(wb, kind, ext, shape):
    phi = _random_phi(shape, ext, 5)
    want = np_symmetrise(phi, ext, kind)
    with wb.Lattice(shape, CD[ext]) as lat:
        lat.set_phi(phi)
        lat.symmetrise_wavefunction(kind)
        got = lat.get_phi()
        assert np.array_equal(_bits(got), _bits(want))
        assert _ring_is_zero(got, ext)
        lat.symmetrise_wavefunction(wb.SYMMETRIES[kind])  # by index: applying it twice = applying it once
        assert np.array_equal(_bits(lat.get_phi()), _bits(want))


@gpu
def test_symmetrise_statuses_and_the_no_op(wb):
    with wb.Lattice((8, 9, 10)) as lat:
        for kind in (0, 2):
            with pytest.raises(wb.WaferError) as ei:
                lat.symmetrise_wavefunction(kind)
            assert ei.value.status == 6  # phi not set yet
        for kind in (-1, 5, 100):
            with pytest.raises(wb.WaferError) as ei:
                lat.symmetrise_wavefunction(kind)
            assert ei.value.status == 1
        phi = _random_phi((8, 9, 10), 1, 3)
        lat.set_phi(phi)
        n = lat.kernel_launches
        lat.symmetrise_wavefunction("NotConstrained")
        assert lat.kernel_launches == n
        assert np.array_equal(_bits(lat.get_phi()), _bits(phi))
        n = lat.kernel_launches  # get_phi launches its pack kernel
        lat.symmetrise_wavefunction("AboutY")
        assert lat.kernel_launches == n + 1
        for sig in (float("nan"), float("inf"), -1.0):
            with pytest.raises(wb.WaferError) as ei:
                lat.set_initial_conditions("Gaussian", sig=sig)
            assert ei.value.status == 1


# ---------------------------------------------------------------------------------------------- GPU: cached check sums
@gpu
@pytest.mark.parametrize("change", ["symmetrise", "gaussian"])
def test_fused_check_sums_are_dropped_by_the_new_calls(wb, oracle, change):
    """evolve(0, >= 64) leaves the point-wise check sums of its last sweep for the next check; after symmetrise or
    generate_gaussian the check must describe the new state, like a context that never fuses them"""
    shape = (22, 35, 61)
    rng = np.random.default_rng(29)
    g = oracle.make_grid(*shape, ext=1, dn=0.1, dt=6.25e-4, mass=1.0)
    v = rng.normal(size=g.padded_shape) * 0.3
    phi = _random_phi(shape, 1, 31)
    checks = []
    for flags in (0, FLAG_NO_FUSED_CHECK):
        with wb.Lattice(shape, dn=g.dn, dt=g.dt, mass=g.mass, flags=flags) as lat:
            lat.set_potential(v)
            lat.set_phi(phi)
            lat.evolve(0, 64)
            if change == "symmetrise":
                state = np_symmetrise(lat.get_phi(), 1, "AntisymAboutZ")
                lat.symmetrise_wavefunction("AntisymAboutZ")
                assert np.array_equal(_bits(lat.get_phi()), _bits(state))
            else:
                lat.set_initial_conditions("Gaussian", sig=0.7, seed=99)
                state = lat.get_phi()
                assert np.abs(state - np_gaussian(shape, 1, 0.7, 99)).max() <= 1e-13 * 0.7
            checks.append(lat.check(0))
    oracle.set_sum_mode(1)
    try:
        want = oracle.observables(g, state, v)
    finally:
        oracle.set_sum_mode(0)
    scale = max(abs(want["energy"]), want["norm2"], abs(want["r2"]))
    for got in checks:
        for key in want:
            assert abs(got[key] - want[key]) <= SUM_TOL * scale, (key, got[key], want[key])


# ---------------------------------------------------------------------------------------------- GPU: sweeps from a mirrored state
@gpu
@pytest.mark.parametrize("flags", [0, 4, 12])
def test_sweeps_from_an_antisymmetric_start_are_bit_exact(wb, oracle, flags):
    """(40, 512, 512): the time-tiled plan on 148 SMs has one x chunk, one round and a statically cut tail"""
    shape = (40, 512, 512)
    rng = np.random.default_rng(41)
    g = oracle.make_grid(*shape, ext=1, dn=0.05, dt=6.25e-4, mass=1.0)
    v = rng.normal(size=g.padded_shape) * 3.0
    a, b = oracle.build_ab(v, g.dt)
    phi = np_symmetrise(oracle.initial_condition(g, "Boolean"), 1, "AntisymAboutZ")
    with wb.Lattice(shape, dn=g.dn, dt=g.dt, mass=g.mass, flags=flags) as lat:
        if flags == 0:
            plan = wb.tb2_plan(shape[1], shape[2], 0, shape[0], lat.device_info()["sm_count"])
            assert (plan[:, 0] >= 0).any()  # a tail
        lat.set_potential(v)
        lat.set_initial_conditions("Boolean")
        lat.symmetrise_wavefunction("AntisymAboutZ")
        assert np.array_equal(_bits(lat.get_phi()), _bits(phi))
        lat.evolve(0, 7)
        got7 = lat.get_phi()
        lat.evolve(0, 6)
        got13 = lat.get_phi()
    oracle.evolve(g, phi, a, b, 7)
    assert np.array_equal(got7, phi)
    oracle.evolve(g, phi, a, b, 6)
    assert np.array_equal(got13, phi)


# ---------------------------------------------------------------------------------------------- GPU: the Gaussian
@gpu
def test_gaussian_is_reproducible_and_scales_with_sig(wb):
    shape = (21, 30, 37)
    with wb.Lattice(shape) as one, wb.Lattice(shape) as two:
        one.set_initial_conditions("Gaussian", sig=1.0, seed=1234)
        two.set_initial_conditions("Gaussian", sig=1.0, seed=1234)
        f1 = one.get_phi()
        assert np.array_equal(_bits(f1), _bits(two.get_phi()))
        two.set_initial_conditions("Gaussian", sig=1.0, seed=1235)
        other = two.get_phi()
        assert np.mean(npr.work(other, 1) != npr.work(f1, 1)) > 0.999
        two.set_initial_conditions("Gaussian", sig=2.0, seed=1234)
        assert np.array_equal(_bits(two.get_phi()), _bits(2.0 * f1))
        two.set_initial_conditions("Gaussian", sig=1.0, seed=1234 + (7 << 32))  # the seed's high word is used too
        assert not np.array_equal(two.get_phi(), f1)


@gpu
@pytest.mark.parametrize("ext", [1, 3])
def test_gaussian_matches_the_numpy_recipe(wb, ext):
    shape = (13, 29, 45)
    for sig, seed in ((1.0, 0), (0.25, 2 ** 64 - 3)):
        want = np_gaussian(shape, ext, sig, seed)
        with wb.Lattice(shape, CD[ext]) as lat:
            lat.set_phi(_random_phi(shape, ext, 1))  # overwritten everywhere
            lat.set_initial_conditions("Gaussian", sig=sig, seed=seed)
            got = lat.get_phi()
        assert np.abs(got - want).max() <= 1e-13 * sig
        assert _ring_is_zero(got, ext)


@gpu
def test_gaussian_statistics_at_128_cubed(wb):
    from scipy import stats
    n, sig = 128, 0.8
    with wb.Lattice((n, n, n)) as lat:
        lat.set_initial_conditions("Gaussian", sig=sig, seed=20261020)
        w = npr.work(lat.get_phi(), 1).ravel()
    N = w.size
    assert abs(w.mean()) < 5 * sig / np.sqrt(N)
    assert abs(w.var() - sig ** 2) < 5 * sig ** 2 * np.sqrt(2.0 / N)
    assert stats.kstest(w, lambda x: stats.norm.cdf(x, loc=0.0, scale=sig)).pvalue > 1e-3


# ---------------------------------------------------------------------------------------------- GPU: the front end
def _harmonic_yaml(symmetry="NotConstrained", extra=()):
    base = open(DEFAULT).read()
    base = base.replace("x: 50", "x: 40").replace("y: 50", "y: 40").replace("z: 50", "z: 40")
    base = base.replace("dn: 0.01", "dn: 0.25").replace("dt: 3e-5", "dt: 0.015").replace("mass: 15.9994", "mass: 1.0")
    base = base.replace("wavemax: 1", "wavemax: 0").replace("tolerance: 1e-4", "tolerance: 1e-9")
    base = base.replace("screen_update: 1000", "screen_update: 100").replace("init_symmetry: NotConstrained",
                                                                             "init_symmetry: " + symmetry)
    for a, b in extra:
        assert a in base
        base = base.replace(a, b)
    return base


def _run(binary, tmp_path, name, text, *args, rc=0):
    (tmp_path / (name + ".yaml")).write_text(text)
    r = subprocess.run([binary, "-c", name + ".yaml", "--output-root", name + ".out", *args], capture_output=True,
                       text=True, cwd=tmp_path, timeout=600)
    assert r.returncode == rc, r.stderr[-2000:]
    rows = [l for l in r.stdout.splitlines() if ROW.match(l)]
    return rows, next((tmp_path / (name + ".out")).iterdir())


@gpu
def test_front_end_converges_in_the_constrained_sector(binary, oracle, tmp_path):
    """40^3 Harmonic (hbar omega = 1): AntisymAboutZ from the Boolean start converges to the lowest state that is odd
    in z, one quantum above the ground state; the oracle solves the same run from the numpy-mirrored start."""
    energy = {}
    for sym in ("NotConstrained", "AntisymAboutZ", "AntisymAboutY", "AboutZ"):
        rows, out = _run(binary, tmp_path, sym, _harmonic_yaml(sym))
        energy[sym] = json.loads((out / "observables_0.json").read_text())["energy"]
    g = oracle.make_grid(40, 40, 40, ext=1, dn=0.25, dt=0.015, mass=1.0)
    v = oracle.potential(g, "Harmonic")
    a, b = oracle.build_ab(v, g.dt)
    phi = np_symmetrise(oracle.initial_condition(g, "Boolean"), 1, "AntisymAboutZ")
    conv, rec = oracle.solve(g, v, a, b, phi, tolerance=1e-9, screen_update=100)
    assert conv
    assert energy["AntisymAboutZ"] == pytest.approx(rec[-1]["E"], rel=1e-9)
    # measured on a B200: 1.4941410106751134, 2.486351320006313 (both Antisym kinds) and 1.4941410106759425 (AboutZ);
    # the quantum is 0.9922 at dn = 0.25
    assert energy["AntisymAboutZ"] - energy["NotConstrained"] == pytest.approx(1.0, rel=0.01)
    assert energy["AntisymAboutY"] == pytest.approx(energy["AntisymAboutZ"], rel=1e-9)
    assert energy["AboutZ"] == pytest.approx(energy["NotConstrained"], rel=1e-10)


@gpu
def test_front_end_snapshots_are_symmetrised(binary, tmp_path):
    """grid.rs:137-139: symmetrise, normalise, then write the partial wavefunction"""
    text = _harmonic_yaml("AntisymAboutZ", [("# max_steps: 50000000", "max_steps: 150"),
                                            ("# snap_update: 10000", "snap_update: 100"),
                                            ("save_wavefns: true", "save_wavefns: false")])
    rows, out = _run(binary, tmp_path, "snap", text, rc=1)  # MaxStep
    assert len(rows) == 3
    w = np.array(json.loads((out / "wavefunction_0_partial.json").read_text())["data"], dtype=np.float64)
    w = w.reshape(40, 40, 40)
    assert np.all(w != 0.0)  # so that the JSON text carries every sign
    assert np.array_equal(_bits(w[..., ::-1]), _bits(-w))


@gpu
def test_front_end_gaussian_start_is_seeded(binary, wb, tmp_path):
    extra = [("init_condition: Boolean", "init_condition: Gaussian"), ("sig: 1.0", "sig: 0.5"),
             ("# max_steps: 50000000", "max_steps: 150")]
    text = _harmonic_yaml("NotConstrained", extra)
    runs = [_run(binary, tmp_path, name, text, *args, rc=1)
            for name, args in (("a", ("--seed", "17")), ("b", ("--seed", "17")), ("c", ("--seed", "18")))]
    (ra, oa), (rb, ob), (rc, oc) = runs
    assert ra == rb and len(ra) == 3
    wa = (oa / "wavefunction_0_partial.json").read_text()
    assert wa == (ob / "wavefunction_0_partial.json").read_text()
    assert rc[0] != ra[0]
    with wb.Lattice((40, 40, 40), dn=0.25, dt=0.015, mass=1.0) as lat:
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Gaussian", sig=0.5, seed=17)
        o = lat.check(0)
    want = "     │%11.3f │%19.10e │%15.5f │%15s │" % (0.0, o["energy"] / o["norm2"], np.sqrt(o["r2"] / o["norm2"]), "--   ")
    assert ra[0] == want


# ---------------------------------------------------------------------------------------------- N > 1 (needs >= 2 GPUs on the box)
@gpu
def test_multi_gpu_gaussian_and_symmetry_equal_single_gpu():
    """torchrun scripts/multigpu_initial_state.py on every GPU of the box (2..8)"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(n, 8)),
           "--master-addr", "127.0.0.1", "--master-port", "29613", os.path.join(ROOT, "scripts", "multigpu_initial_state.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"]
