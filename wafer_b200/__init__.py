"""wafer_b200 — host-side mirror of Wafer's hot-path interface over the sm_100a C-ABI library.

`Lattice` keeps the reference's function names and argument meaning (src/grid.rs):
compute_observables, get_norm_squared, normalise_wavefunction, orthogonalise_wavefunction, evolve, solve.
Arrays are numpy float64 in the reference's padded Array3 layout.  Every call goes through
wafer_b200/libwafer_b200.so (include/wafer_b200.h); nothing here computes on the CPU.
"""
import ctypes as C
import os

import numpy as np

from . import _capi
from ._capi import LoadStats, Observables, Params, Record, WriteStats

__all__ = ["Lattice", "slab_partition", "tb2_plan", "WaferError", "POTENTIALS", "INITIAL_CONDITIONS", "SYMMETRIES", "EXT",
           "nccl_unique_id", "pinned_empty", "pin", "unpin", "FLAG_AB_ARRAYS", "FILE_TYPES"]

# PotentialType (config.rs:74-104), InitialCondition (config.rs:153-170), SymmetryConstraint (config.rs:186-197),
# CentralDifference.ext() (config.rs:232-238)
POTENTIALS = {
    "NoPotential": 0, "Cube": 1, "QuadWell": 2, "Periodic": 3, "Coulomb": 4, "ComplexCoulomb": 5,
    "ElipticalCoulomb": 6, "SimpleCornell": 7, "FullCornell": 8, "Harmonic": 9, "ComplexHarmonic": 10,
    "Dodecahedron": 11, "FromFile": 12, "FromScript": 13, "PoschlTeller": 100,
}
FILE_TYPES = {"Messagepack": 0, "Csv": 1, "Json": 2}
INITIAL_CONDITIONS = {"FromFile": 0, "Gaussian": 1, "Coulomb": 2, "Constant": 3, "Boolean": 4}
SYMMETRIES = {"NotConstrained": 0, "AboutZ": 1, "AntisymAboutZ": 2, "AboutY": 3, "AntisymAboutY": 4}
EXT = {"ThreePoint": 1, "FivePoint": 2, "SevenPoint": 3}
FLAG_AB_ARRAYS = 0x1
FLAG_SIMPLE_SWEEP = 0x4
FLAG_TMA_ONE_STEP = 0x8

_STATUS = {1: "INVALID", 2: "NO_DEVICE", 3: "CUDA", 4: "NCCL", 5: "RING_NONZERO", 6: "NOT_READY", 7: "MAX_STEP",
           8: "NONFINITE", 9: "IO", 10: "FORMAT"}
_dp = C.POINTER(C.c_double)


class WaferError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("wafer_b200: %s (%d): %s" % (_STATUS.get(status, "?"), status, message))
        self.status = status


def slab_partition(nx, world, rank):
    """work x-planes [x0, x1) owned by `rank` of `world` (wafer_slab_partition; pure host arithmetic)"""
    x0, x1 = C.c_uint64(), C.c_uint64()
    rc = _capi.load().wafer_slab_partition(nx, world, rank, C.byref(x0), C.byref(x1))
    if rc:
        raise WaferError(rc, "wafer_slab_partition(%d, %d, %d)" % (nx, world, rank))
    return x0.value, x1.value


def tb2_plan(ny, nz, xb, xe, slots=148):
    """work distribution of the time-tiled sweep (wafer_tb2_plan): array of rows [owner, y0, z0, xa, xz]"""
    lib = _capi.load()
    n = C.c_uint64()
    rc = lib.wafer_tb2_plan(ny, nz, xb, xe, slots, None, 0, C.byref(n))
    if rc:
        raise WaferError(rc, "wafer_tb2_plan(%d, %d, %d, %d, %d)" % (ny, nz, xb, xe, slots))
    out = np.zeros((n.value, 5), dtype=np.int32)
    rc = lib.wafer_tb2_plan(ny, nz, xb, xe, slots, out.ctypes.data_as(C.POINTER(C.c_int32)), n.value, C.byref(n))
    if rc:
        raise WaferError(rc, "wafer_tb2_plan")
    return out


def nccl_unique_id():
    """128-byte ncclUniqueId; rank 0 makes it, the harness broadcasts it (torch.distributed / MPI / a file)."""
    buf = (C.c_uint8 * 128)()
    rc = _capi.load().wafer_nccl_unique_id(buf)
    if rc:
        raise WaferError(rc, _capi.load().wafer_last_error(None).decode())
    return bytes(buf)


def pinned_empty(shape):
    """float64 array in page-locked host memory (wafer_host_alloc), for full-speed host<->device copies."""
    lib = _capi.load()
    n = int(np.prod(shape))
    p = C.c_void_p()
    rc = lib.wafer_host_alloc(C.byref(p), n * 8)
    if rc:
        raise WaferError(rc, "wafer_host_alloc(%d bytes) failed" % (n * 8))
    buf = (C.c_double * n).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.float64).reshape(shape)
    _PINNED[arr.ctypes.data] = p
    return arr


_PINNED = {}


def pinned_free(arr):
    """Release a pinned_empty() array; the array (and every view of it) must not be used afterwards."""
    _capi.load().wafer_host_free(_PINNED.pop(arr.ctypes.data))


def pin(arr):
    """page-lock an existing C-contiguous float64 array in place (wafer_host_register); undo with unpin()"""
    rc = _capi.load().wafer_host_register(arr.ctypes.data_as(C.c_void_p), arr.nbytes)
    if rc:
        raise WaferError(rc, "wafer_host_register(%d bytes) failed" % arr.nbytes)
    return arr


def unpin(arr):
    _capi.load().wafer_host_unregister(arr.ctypes.data_as(C.c_void_p))


def _p(a):
    if not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]):
        raise TypeError("expected a C-contiguous float64 ndarray (the reference's Array3<R64> memory)")
    return a.ctypes.data_as(_dp)


class Lattice:
    """One GPU's slab of the lattice: Config.grid + central_difference + mass, Potentials and phi on the device."""

    def __init__(self, size, central_difference="ThreePoint", dn=0.01, dt=3e-5, mass=1.0, device=-1, rank=0, world=1,
                 nccl_id=None, flags=0):
        self._lib = _capi.load()
        self._h = C.c_void_p()
        ext = EXT[central_difference] if isinstance(central_difference, str) else int(central_difference)
        self.size, self.ext, self.dn, self.dt, self.mass = tuple(int(s) for s in size), ext, dn, dt, mass
        idbuf = None
        if nccl_id is not None:
            idbuf = (C.c_uint8 * 128).from_buffer_copy(nccl_id)
        p = Params(self.size[0], self.size[1], self.size[2], ext, dn, dt, mass, device, rank, world,
                   C.cast(idbuf, C.POINTER(C.c_uint8)) if idbuf is not None else None, 0, flags)
        rc = self._lib.wafer_create(C.byref(p), C.byref(self._h))
        if rc:
            self._h = C.c_void_p()
            raise WaferError(rc, self._lib.wafer_last_error(None).decode())
        self.rank, self.world = rank, world

    # ---- plumbing
    def _ck(self, rc):
        if rc:
            raise WaferError(rc, self._lib.wafer_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.wafer_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def padded_shape(self):
        e = self.ext
        return tuple(s + 2 * e for s in self.size)

    @property
    def slab(self):
        x0, x1 = C.c_uint64(), C.c_uint64()
        self._ck(self._lib.wafer_slab(self._h, C.byref(x0), C.byref(x1)))
        return x0.value, x1.value

    def synchronize(self):
        self._ck(self._lib.wafer_synchronize(self._h))

    def timer_begin(self):
        self._ck(self._lib.wafer_timer_begin(self._h))

    def timer_end(self):
        ms = C.c_double()
        self._ck(self._lib.wafer_timer_end(self._h, C.byref(ms)))
        return ms.value

    @property
    def kernel_launches(self):
        return int(self._lib.wafer_kernel_launches(self._h))

    @property
    def sweep_variant(self):
        return self._lib.wafer_sweep_variant(self._h).decode()

    def p2p_export(self):
        """192-byte blob (CUDA IPC handles) the x-neighbours need for the fused halo path"""
        buf = (C.c_uint8 * 192)()
        self._ck(self._lib.wafer_p2p_export(self._h, buf))
        return bytes(buf)

    def p2p_connect(self, lower, upper):
        """lower / upper: p2p_export() blobs of rank-1 / rank+1 (None at the ends of the chain)"""
        lo = (C.c_uint8 * 192).from_buffer_copy(lower) if lower is not None else None
        hi = (C.c_uint8 * 192).from_buffer_copy(upper) if upper is not None else None
        self._ck(self._lib.wafer_p2p_connect(self._h, lo, hi))

    def selftest_division(self, den, n=1 << 24, seed=0):
        bad = C.c_uint64()
        self._ck(self._lib.wafer_selftest_division(self._h, den, n, seed, C.byref(bad)))
        return bad.value

    def device_info(self):
        name = C.create_string_buffer(256)
        sm, ma, mi, mem = C.c_int32(), C.c_int32(), C.c_int32(), C.c_uint64()
        self._ck(self._lib.wafer_device_info(self._h, name, 256, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem)))
        return dict(name=name.value.decode(), sm_count=sm.value, cc=(ma.value, mi.value), mem_bytes=mem.value)

    # ---- Potentials (potential.rs:14-25, 75-175)
    def set_potential(self, v):
        assert v.shape == self.padded_shape
        self._ck(self._lib.wafer_set_potential(self._h, _p(v)))

    def get_potential(self):
        out = np.zeros(self.padded_shape)
        self._ck(self._lib.wafer_get_potential(self._h, _p(out)))
        return out

    def generate_potential(self, kind, sig=1.0):
        self._ck(self._lib.wafer_generate_potential(self._h, POTENTIALS[kind] if isinstance(kind, str) else kind, sig))

    def set_pot_sub(self, pot_sub):
        """pot_sub like Potentials.pot_sub: None, a scalar, or a work-sized array."""
        if pot_sub is None:
            self._ck(self._lib.wafer_set_pot_sub_scalar(self._h, 0.0))
        elif isinstance(pot_sub, np.ndarray):
            assert pot_sub.shape == self.size
            self._ck(self._lib.wafer_set_pot_sub_array(self._h, _p(pot_sub)))
        else:
            self._ck(self._lib.wafer_set_pot_sub_scalar(self._h, float(pot_sub)))

    # ---- phi and w_store
    def set_phi(self, phi):
        assert phi.shape == self.padded_shape
        self._ck(self._lib.wafer_set_phi(self._h, _p(phi)))

    def get_phi(self, out=None):
        out = np.zeros(self.padded_shape) if out is None else out
        self._ck(self._lib.wafer_get_phi(self._h, _p(out)))
        return out

    def slab_planes(self, which):
        """padded x-planes [p0,p1) of the global array that set_phi_slab reads (which=0) / get_phi_slab writes (1)"""
        p0, p1 = C.c_uint64(), C.c_uint64()
        self._ck(self._lib.wafer_slab_planes(self._h, which, C.byref(p0), C.byref(p1)))
        return p0.value, p1.value

    def set_phi_slab(self, chunk):
        p0, p1 = self.slab_planes(0)
        assert chunk.shape == (p1 - p0,) + self.padded_shape[1:]
        self._ck(self._lib.wafer_set_phi_slab(self._h, _p(chunk)))

    def get_phi_slab(self, out=None):
        p0, p1 = self.slab_planes(1)
        out = np.zeros((p1 - p0,) + self.padded_shape[1:]) if out is None else out
        assert out.shape == (p1 - p0,) + self.padded_shape[1:]
        self._ck(self._lib.wafer_get_phi_slab(self._h, _p(out)))
        return out

    def set_phi_owned(self, chunk):
        """inverse of get_phi_slab: owned planes in, ghost planes fetched from the neighbours (collective)"""
        p0, p1 = self.slab_planes(1)
        assert chunk.shape == (p1 - p0,) + self.padded_shape[1:]
        self._ck(self._lib.wafer_set_phi_owned(self._h, _p(chunk)))

    def phi_checksum(self, x_begin=0, x_end=None):
        """(wrapping sum, xor) of the per-site hashes of global work planes [x_begin, x_end) owned by this rank"""
        out = (C.c_uint64 * 2)()
        self._ck(self._lib.wafer_phi_checksum(self._h, x_begin, self.size[0] if x_end is None else x_end, out))
        return int(out[0]), int(out[1])

    def debug_halo_delay(self, nanoseconds):
        """fault injection: stall this rank's halo stream before every boundary pass (tests of the GPU-GPU ordering)"""
        self._ck(self._lib.wafer_debug_halo_delay(self._h, int(nanoseconds)))

    def set_initial_conditions(self, kind, sig=1.0, seed=0):
        """config::set_initial_conditions (config.rs:577-627) evaluated on the device.  "Gaussian" is N(0, sig) at every
        work site from a counter-based generator keyed by `seed` (wafer_generate_gaussian): reproducible, and the same
        at any world size; sig and seed are unused by the other kinds."""
        k = INITIAL_CONDITIONS[kind] if isinstance(kind, str) else int(kind)
        if k == INITIAL_CONDITIONS["Gaussian"]:
            self._ck(self._lib.wafer_generate_gaussian(self._h, float(sig), int(seed)))
        else:
            self._ck(self._lib.wafer_generate_initial_condition(self._h, k))

    def symmetrise_wavefunction(self, kind):
        """config::symmetrise_wavefunction (config.rs:691-728) on the device: kind is a SYMMETRIES name or index.
        Mirrors the work area about its centre in y or z, copying the lower half (negated for the Antisym kinds)."""
        self._ck(self._lib.wafer_symmetrise(self._h, SYMMETRIES[kind] if isinstance(kind, str) else int(kind)))

    # ---- input files resampled on the device: fill_data (input.rs:149-176) / read_csv (input.rs:641-657)
    def _resampled(self, fn, arr, from_csv):
        if arr.ndim != 3:
            raise ValueError("expected a 3-D array (the array of an input file), got shape %r" % (arr.shape,))
        sx, sy, sz = arr.shape
        self._ck(fn(self._h, _p(arr), sx, sy, sz, 1 if from_csv else 0))

    def set_phi_resampled(self, arr, from_csv=False):
        """phi from the WORK-area array of an input file as read, shape (sx, sy, sz): trilinear resample on the
        reference's padded-size basis (Messagepack / Json, from_csv=False, always resampled; a padded-size array is
        refused), or for from_csv=True a straight copy of a work-sized array.  Runs on the device."""
        self._resampled(self._lib.wafer_set_phi_resampled, arr, from_csv)

    def set_potential_resampled(self, arr, from_csv=False):
        """V from an input file's array, resampled like set_phi_resampled (the FromFile potential)"""
        self._resampled(self._lib.wafer_set_potential_resampled, arr, from_csv)

    def push_lower_resampled(self, arr, from_csv=False):
        """w_store.push of an input file's array, resampled like set_phi_resampled (input::load_wavefunctions)"""
        self._resampled(self._lib.wafer_push_lower_resampled, arr, from_csv)

    def push_lower(self, q=None):
        """w_store.push(q); with q=None pushes the current phi (grid.rs:241)."""
        if q is None:
            self._ck(self._lib.wafer_push_lower_from_phi(self._h))
        else:
            self._ck(self._lib.wafer_push_lower(self._h, _p(q)))

    def get_lower(self, idx):
        out = np.zeros(self.padded_shape)
        self._ck(self._lib.wafer_get_lower(self._h, idx, _p(out)))
        return out

    def phi_from_lower(self, idx):
        self._ck(self._lib.wafer_phi_from_lower(self._h, idx))

    def phi_seed_from_lower(self, idx):
        """deterministic excited-state start: phi = w_store[idx] * seed polynomial (see generators.cuh)"""
        self._ck(self._lib.wafer_phi_seed_from_lower(self._h, idx))

    def clear_lowers(self):
        self._ck(self._lib.wafer_clear_lowers(self._h))

    @property
    def num_lowers(self):
        return int(self._lib.wafer_num_lowers(self._h))

    # ---- array files: output::wavefunction / output::potential (output.rs:79-216), encoded on the device
    def write_array(self, what, path, file_type):
        """Write the work area of psi (what="phi" or 0) or V ("potential" or 1) to `path` (extension included) as
        file_type "Messagepack" / "Csv" / "Json" (or 0 / 1 / 2), byte for byte the front end's formats.hpp writers.
        Collective when world > 1: every rank passes the same path and writes its planes into the one file.
        Returns dict(bytes=this rank's bytes, file_bytes=size of the file, host_formatted=sites formatted on the host)."""
        w = {"phi": 0, "potential": 1}[what] if isinstance(what, str) else int(what)
        ft = FILE_TYPES[file_type] if isinstance(file_type, str) else int(file_type)
        st = WriteStats()
        self._ck(self._lib.wafer_write_array(self._h, w, ft, os.fsencode(path), C.byref(st)))
        return dict(bytes=st.bytes, file_bytes=st.file_bytes, host_formatted=st.host_formatted)

    def load_array(self, what, path, file_type):
        """Decode the array file `path` on the device into psi (what="phi" or 0), V ("potential" or 1) or a new lower
        state ("lower" or 2), as set_phi_resampled / set_potential_resampled / push_lower_resampled of the array the
        front end's formats.hpp reader returns (from_csv for "Csv"), bit for bit.  file_type: "Messagepack" / "Csv" /
        "Json" (or 0 / 1 / 2).  Raises WaferError with status 10 (FORMAT), nothing changed, for a file not in the
        canonical layout of the host writers.  Returns dict(sx, sy, sz, bytes_read, sites_converted, host_converted)."""
        w = {"phi": 0, "potential": 1, "lower": 2}[what] if isinstance(what, str) else int(what)
        ft = FILE_TYPES[file_type] if isinstance(file_type, str) else int(file_type)
        st = LoadStats()
        self._ck(self._lib.wafer_load_array(self._h, w, ft, os.fsencode(path), C.byref(st)))
        return dict(sx=st.sx, sy=st.sy, sz=st.sz, bytes_read=st.bytes_read, sites_converted=st.sites_converted,
                    host_converted=st.host_converted)

    # ---- the hot path, reference names (grid.rs)
    def compute_observables(self):
        o = Observables()
        self._ck(self._lib.wafer_observables_compute(self._h, C.byref(o)))
        return dict(energy=o.energy, norm2=o.norm2, v_infinity=o.v_infinity, r2=o.r2)

    def get_norm_squared(self):
        out = C.c_double()
        self._ck(self._lib.wafer_norm2(self._h, C.byref(out)))
        return out.value

    def normalise_wavefunction(self, norm2):
        self._ck(self._lib.wafer_normalise(self._h, norm2))

    def orthogonalise_wavefunction(self, wnum):
        self._ck(self._lib.wafer_orthogonalise(self._h, wnum))

    def evolve(self, wnum, steps):
        self._ck(self._lib.wafer_evolve(self._h, wnum, steps))

    def check(self, wnum):
        o = Observables()
        self._ck(self._lib.wafer_check(self._h, wnum, C.byref(o)))
        return dict(energy=o.energy, norm2=o.norm2, v_infinity=o.v_infinity, r2=o.r2)

    def solve(self, wnum, tolerance, max_steps=None, screen_update=1000, snap_update=None, max_records=4096):
        """grid.rs:50-246.  Returns (converged, records); raises on anything but OK / MAX_STEP."""
        recs = (Record * max_records)()
        n = C.c_uint64()
        rc = self._lib.wafer_solve(self._h, wnum, tolerance, -1 if max_steps is None else int(max_steps),
                                   screen_update, 0 if snap_update is None else int(snap_update), recs, max_records,
                                   C.byref(n))
        if rc not in (0, 7):
            self._ck(rc)
        out = []
        for i in range(min(n.value, max_records)):
            r = recs[i]
            out.append(dict(step=r.step, tau=r.tau, diff=r.diff, energy=r.obs.energy, norm2=r.obs.norm2,
                            v_infinity=r.obs.v_infinity, r2=r.obs.r2, E=r.obs.energy / r.obs.norm2))
        return rc == 0, out
