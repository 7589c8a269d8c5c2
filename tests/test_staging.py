"""The host <-> device staging ring shared by set_phi / get_phi (upload, download), the resampling entries and the
array files (wafer_write_array, wafer_load_array).  Its slots are sized by the first user and grown by later ones:
here a resample from a large source grows them on a small lattice, and every other user then runs on the grown
slots, in both orders.  Each operation must give, bit for bit and byte for byte, what it gives on a fresh context."""
import numpy as np
import pytest

gpu = pytest.mark.gpu

N = (40, 40, 40)  # SevenPoint: 880 KB slots, less than two x-planes of a 256^3 source (1 MB)
FORMATS = {0: "mpk", 1: "csv", 2: "json"}


@pytest.fixture(scope="module")
def wb():
    import wafer_b200
    return wafer_b200


def _lattice(wb):
    return wb.Lattice(N, "SevenPoint", dn=0.1, dt=1e-3, mass=1.0)


def _bits(x):  # a file's bytes, or an array's shape and bits
    return x if isinstance(x, bytes) else (x.shape, x.tobytes())


def _src(shape, seed):
    return np.random.default_rng(seed).normal(size=shape) + 0.5


@gpu
def test_users_of_the_ring_in_turn_on_one_context(wb, tmp_path):
    big, small = _src((256, 256, 256), 3), _src((30, 20, 25), 4)
    with _lattice(wb) as lat:  # the files every load reads
        lat.set_phi_resampled(big)
        files = {ft: tmp_path / ("in.%s" % ext) for ft, ext in FORMATS.items()}
        for ft, path in files.items():
            lat.write_array("phi", str(path), ft)

    def resample_big(lat, tag):
        lat.set_phi_resampled(big)
        return [lat.get_phi()]

    def write(lat, tag):
        out = []
        for ft, ext in FORMATS.items():
            path = tmp_path / ("%s.%s" % (tag, ext))
            lat.write_array("phi", str(path), ft)
            out.append(path.read_bytes())
        return out

    def load(lat, tag):
        out = []
        for ft, path in files.items():
            lat.load_array("phi", str(path), ft)
            out.append(lat.get_phi())
        return out

    def get_set(lat, tag):
        phi = lat.get_phi()
        lat.set_phi(phi)
        return [phi, lat.get_phi(), lat.get_phi_slab()]

    def resample_small(lat, tag):
        lat.set_phi_resampled(small)
        return [lat.get_phi()]

    ops = [(resample_big, False), (write, True), (load, False), (get_set, True), (resample_small, False)]
    for order, seq in (("forward", ops), ("reverse", ops[::-1])):
        with _lattice(wb) as lat:
            for k, (op, needs_phi) in enumerate(seq):
                phi = lat.get_phi() if needs_phi else None
                got = op(lat, "%s%d" % (order, k))
                with _lattice(wb) as fresh:
                    if needs_phi:
                        fresh.set_phi(phi)
                    want = op(fresh, "%s%d_fresh" % (order, k))
                assert len(got) == len(want)
                for i, (g, w) in enumerate(zip(got, want)):
                    assert _bits(g) == _bits(w), (order, op.__name__, i)
