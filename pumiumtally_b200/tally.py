"""Python host-side mirror of ``pumitally::PumiTally`` over the C ABI.

Same method names and argument meaning as the reference class
(reference: src/pumitally/PumiTally.h:50-103) so parity tests read like the
reference's own test (test/test_pumi_tally_impl_methods.cpp).  Every call goes
through ``libpumitally.so`` (include/pumitally_c.h); there is no Python or CPU
implementation of the path behind this class -- if the CUDA library is missing
or no GPU is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
# PUMITALLY_LIB selects another build of the same library (tests of the measured alternative kernels
# use lib/libpumitally_exp.so); the default is the product library.
LIB_PATH = os.environ.get("PUMITALLY_LIB") or os.path.join(_PKG, "lib", "libpumitally.so")
_lib = None

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_bp = C.POINTER(C.c_int8)
_u8p = C.POINTER(C.c_uint8)


class Stats(C.Structure):
    _fields_ = [
        ("segments", C.c_uint64), ("tracks", C.c_uint64), ("relocations", C.c_uint64),
        ("lost", C.c_uint64), ("moves", C.c_uint64), ("kernel_ms", C.c_double),
        ("h2d_bytes", C.c_double), ("plane_fallbacks", C.c_uint64),
    ]


# name -> (restype, argtypes); also the list tests check against include/pumitally_c.h
C_API = {
    "pumitally_create": (C.c_void_p, [C.c_char_p, C.c_int32, C.POINTER(C.c_int), C.c_void_p]),
    "pumitally_copy_initial_position": (C.c_int, [C.c_void_p, _dp, C.c_int32]),
    "pumitally_move_to_next_location": (C.c_int, [C.c_void_p, _dp, _dp, _bp, _dp, C.c_int32]),
    "pumitally_move_to_next_location_binned": (C.c_int, [C.c_void_p, _dp, _dp, _bp, _dp, _ip, C.c_int32]),
    "pumitally_move_to_next_location_device_binned": (
        C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pumitally_set_score_bins": (C.c_int, [C.c_void_p, C.c_int32]),
    "pumitally_get_score_bins": (C.c_int32, [C.c_void_p]),
    "pumitally_write_tally_results": (C.c_int, [C.c_void_p]),
    "pumitally_destroy": (None, [C.c_void_p]),
    "pumitally_create_from_arrays": (C.c_void_p, [_dp, C.c_int64, _ip, C.c_int64, C.c_int32, C.c_int32]),
    "pumitally_num_elements": (C.c_int64, [C.c_void_p]),
    "pumitally_num_particles": (C.c_int32, [C.c_void_p]),
    "pumitally_get_flux": (C.c_int, [C.c_void_p, _dp, C.c_int64]),
    "pumitally_get_normalized_flux": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int64]),
    "pumitally_get_element_ids": (C.c_int, [C.c_void_p, _ip, C.c_int64]),
    "pumitally_get_positions": (C.c_int, [C.c_void_p, _dp, C.c_int64]),
    "pumitally_get_adjacency": (C.c_int, [C.c_void_p, _ip, C.c_int64]),
    "pumitally_reset_tally": (C.c_int, [C.c_void_p]),
    "pumitally_set_source_normalization": (C.c_int, [C.c_void_p, C.c_int32, C.c_double]),
    "pumitally_get_source_normalization": (C.c_double, [C.c_void_p]),
    "pumitally_get_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "pumitally_set_output_name": (C.c_int, [C.c_void_p, C.c_char_p]),
    "pumitally_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "pumitally_get_option": (C.c_int64, [C.c_void_p, C.c_char_p]),
    "pumitally_copy_initial_position_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pumitally_move_to_next_location_device": (
        C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pumitally_set_state_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "pumitally_get_state_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "pumitally_get_flux_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "pumitally_flux_device_ptr": (C.c_void_p, [C.c_void_p]),
    "pumitally_synchronize": (C.c_int, [C.c_void_p]),
    "pumitally_nccl_unique_id": (C.c_int, [_u8p]),
    "pumitally_comm_init": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, _u8p]),
    "pumitally_allreduce_tally": (C.c_int, [C.c_void_p]),
    "pumitally_reduce_tally_to_owners": (C.c_int, [C.c_void_p]),
    "pumitally_exchange_tally": (C.c_int, [C.c_void_p]),
    "pumitally_end_batch": (C.c_int, [C.c_void_p]),
    "pumitally_get_tally_statistics": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int64]),
    "pumitally_get_max_relative_error": (
        C.c_int, [C.c_void_p, C.c_double, _dp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "pumitally_debug_order": (C.c_int64, [C.c_void_p, _ip, C.c_int64]),
    "pumitally_debug_stage": (C.c_int64, [_dp, _dp, _bp, _dp, _dp, _dp, _bp, C.c_int64, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_int64]),
    "pumitally_version": (C.c_char_p, []),
}


def load_library():
    """dlopen libpumitally.so and declare the C ABI. Raises if it was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`."
                " There is no CPU implementation of the tally path in this package.")
        L = C.CDLL(LIB_PATH)
        for name, (rt, at) in C_API.items():
            fn = getattr(L, name)
            fn.restype = rt
            fn.argtypes = at
        _lib = L
    return _lib


def _host_f64(a, what):
    a = np.asarray(a)
    if a.dtype != np.float64 or not a.flags.c_contiguous:
        a = np.ascontiguousarray(a, dtype=np.float64)
    return a.reshape(-1)


class PumiTally:
    """Track-length tally engine on one B200.

    ``PumiTally(mesh_filename, num_particles)`` follows the reference constructor;
    ``PumiTally.from_arrays(coords, tet2vert, num_particles)`` takes the mesh in memory.
    """

    def __init__(self, mesh_filename: str, num_particles: int, argv=None, _handle=None):
        self._L = load_library()
        self.num_particles = int(num_particles)
        if _handle is None:
            argc = C.c_int(0)
            _handle = self._L.pumitally_create(str(mesh_filename).encode(), self.num_particles,
                                               C.byref(argc), None)
        if not _handle:
            raise RuntimeError("pumitally engine construction failed (mesh unreadable or no CUDA device)")
        self._h = C.c_void_p(_handle)
        self.num_elements = int(self._L.pumitally_num_elements(self._h))

    @classmethod
    def from_spec(cls, mesh_filename: str, num_particles: int, device: int = -1):
        """Reference constructor with the CUDA device passed the way the reference passes
        runtime options: through argv (``--pumitally-device=<id>``)."""
        L = load_library()
        args = [b"pumitally"] + ([f"--pumitally-device={device}".encode()] if device >= 0 else [])
        argv = (C.c_char_p * (len(args) + 1))(*args, None)
        argc = C.c_int(len(args))
        argv_p = C.cast(argv, C.POINTER(C.c_char_p))
        h = L.pumitally_create(str(mesh_filename).encode(), int(num_particles), C.byref(argc), C.byref(argv_p))
        if not h:
            raise RuntimeError("pumitally engine construction failed (mesh unreadable or no CUDA device)")
        return cls("", num_particles, _handle=h)

    @classmethod
    def from_arrays(cls, coords, tet2vert, num_particles: int, device: int = -1):
        L = load_library()
        coords = np.ascontiguousarray(coords, dtype=np.float64)
        t2v = np.ascontiguousarray(tet2vert, dtype=np.int32)
        h = L.pumitally_create_from_arrays(coords.ctypes.data_as(_dp), coords.shape[0],
                                           t2v.ctypes.data_as(_ip), t2v.shape[0],
                                           int(num_particles), int(device))
        if not h:
            raise RuntimeError("pumitally engine construction failed (bad mesh or no CUDA device)")
        return cls("", num_particles, _handle=h)

    def close(self):
        if getattr(self, "_h", None):
            self._L.pumitally_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- reference interface -------------------------------------------------
    def CopyInitialPosition(self, init_particle_positions, size=None):
        xyz = _host_f64(init_particle_positions, "init_particle_positions")
        size = xyz.size if size is None else int(size)
        if self._L.pumitally_copy_initial_position(self._h, xyz.ctypes.data_as(_dp), size):
            raise RuntimeError("CopyInitialPosition failed")

    def MoveToNextLocation(self, particle_origin, particle_destinations, flying, weights, size=None):
        o = _host_f64(particle_origin, "particle_origin")
        d = _host_f64(particle_destinations, "particle_destinations")
        w = _host_f64(weights, "weights")
        if not (isinstance(flying, np.ndarray) and flying.dtype == np.int8 and flying.flags.c_contiguous):
            raise TypeError("flying must be a contiguous int8 numpy array (the engine zeroes it)")
        size = o.size if size is None else int(size)
        if self._L.pumitally_move_to_next_location(self._h, o.ctypes.data_as(_dp), d.ctypes.data_as(_dp),
                                                   flying.ctypes.data_as(_bp), w.ctypes.data_as(_dp), size):
            raise RuntimeError("MoveToNextLocation failed")

    # ---- score filter ----------------------------------------------------------
    def set_score_bins(self, nbins: int):
        """nbins flux arrays (resets the tally); binned moves score particle i into array bins[i]."""
        if self._L.pumitally_set_score_bins(self._h, int(nbins)):
            raise ValueError(f"set_score_bins({nbins}) failed")

    @property
    def score_bins(self) -> int:
        return int(self._L.pumitally_get_score_bins(self._h))

    def MoveToNextLocationBinned(self, particle_origin, particle_destinations, flying, weights, bins, size=None):
        o = _host_f64(particle_origin, "particle_origin")
        d = _host_f64(particle_destinations, "particle_destinations")
        w = _host_f64(weights, "weights")
        if not (isinstance(flying, np.ndarray) and flying.dtype == np.int8 and flying.flags.c_contiguous):
            raise TypeError("flying must be a contiguous int8 numpy array (the engine zeroes it)")
        if not (isinstance(bins, np.ndarray) and bins.dtype == np.int32 and bins.flags.c_contiguous and bins.size == w.size):
            raise TypeError("bins must be a contiguous int32 numpy array, one entry per particle")
        size = o.size if size is None else int(size)
        if self._L.pumitally_move_to_next_location_binned(self._h, o.ctypes.data_as(_dp), d.ctypes.data_as(_dp),
                                                          flying.ctypes.data_as(_bp), w.ctypes.data_as(_dp),
                                                          bins.ctypes.data_as(_ip), size):
            raise RuntimeError("MoveToNextLocationBinned failed")

    def move_device_binned(self, d_origin, d_dest, d_flying, d_weights, d_bins, stream=None):
        if self._L.pumitally_move_to_next_location_device_binned(self._h, d_origin, d_dest, d_flying, d_weights, d_bins,
                                                                 3 * self.num_particles, stream):
            raise RuntimeError("MoveToNextLocationBinned(device) failed")

    @property
    def flux_bins(self):
        """Raw flux of every score bin: array [nbins, num_elements]."""
        out = np.empty((self.score_bins, self.num_elements))
        if self._L.pumitally_get_flux(self._h, out.ctypes.data_as(_dp), out.size):
            raise RuntimeError("get_flux failed")
        return out

    def normalized_flux_bins(self):
        f, v = np.empty((self.score_bins, self.num_elements)), np.empty(self.num_elements)
        if self._L.pumitally_get_normalized_flux(self._h, f.ctypes.data_as(_dp), v.ctypes.data_as(_dp), f.size):
            raise RuntimeError("get_normalized_flux failed")
        return f, v

    def WriteTallyResults(self, filename=None):
        if filename is not None:
            self._L.pumitally_set_output_name(self._h, str(filename).encode())
        if self._L.pumitally_write_tally_results(self._h):
            raise RuntimeError("WriteTallyResults failed")

    # ---- raw-pointer variants (host pinned buffers / device tensors) -----------
    def move_host_ptr(self, origin_ptr, dest_ptr, flying_ptr, weights_ptr):
        """MoveToNextLocation on raw host addresses (e.g. pinned torch tensors)."""
        rc = self._L.pumitally_move_to_next_location(
            self._h, C.cast(origin_ptr, _dp), C.cast(dest_ptr, _dp), C.cast(flying_ptr, _bp),
            C.cast(weights_ptr, _dp), 3 * self.num_particles)
        if rc:
            raise RuntimeError("MoveToNextLocation failed")

    def copy_initial_position_device(self, d_xyz_ptr, stream=None):
        if self._L.pumitally_copy_initial_position_device(self._h, d_xyz_ptr, 3 * self.num_particles, stream):
            raise RuntimeError("CopyInitialPosition(device) failed")

    def move_device(self, d_origin, d_dest, d_flying, d_weights, stream=None):
        """MoveToNextLocation on device addresses; enqueues on ``stream`` and returns."""
        if self._L.pumitally_move_to_next_location_device(self._h, d_origin, d_dest, d_flying, d_weights,
                                                          3 * self.num_particles, stream):
            raise RuntimeError("MoveToNextLocation(device) failed")

    def set_state_device(self, d_xyz, d_elem, first, count, stream=None):
        if self._L.pumitally_set_state_device(self._h, d_xyz, d_elem, int(first), int(count), stream):
            raise RuntimeError("set_state_device failed")

    def get_state_device(self, d_xyz, d_elem, first, count, stream=None):
        if self._L.pumitally_get_state_device(self._h, d_xyz, d_elem, int(first), int(count), stream):
            raise RuntimeError("get_state_device failed")

    def get_flux_device(self, d_out, stream=None):
        if self._L.pumitally_get_flux_device(self._h, d_out, stream):
            raise RuntimeError("get_flux_device failed")

    def synchronize(self):
        self._L.pumitally_synchronize(self._h)

    # ---- accessors -----------------------------------------------------------
    @property
    def flux(self):
        out = np.empty(self.num_elements)
        if self._L.pumitally_get_flux(self._h, out.ctypes.data_as(_dp), out.size):
            raise RuntimeError("get_flux failed")
        return out

    def normalized_flux(self):
        f, v = np.empty(self.num_elements), np.empty(self.num_elements)
        if self._L.pumitally_get_normalized_flux(self._h, f.ctypes.data_as(_dp), v.ctypes.data_as(_dp), f.size):
            raise RuntimeError("get_normalized_flux failed")
        return f, v

    @property
    def elem_ids(self):
        out = np.empty(self.num_particles, dtype=np.int32)
        if self._L.pumitally_get_element_ids(self._h, out.ctypes.data_as(_ip), out.size):
            raise RuntimeError("get_element_ids failed")
        return out

    @property
    def positions(self):
        out = np.empty((self.num_particles, 3))
        if self._L.pumitally_get_positions(self._h, out.ctypes.data_as(_dp), out.size):
            raise RuntimeError("get_positions failed")
        return out

    @property
    def adjacency(self):
        out = np.empty((self.num_elements, 4), dtype=np.int32)
        if self._L.pumitally_get_adjacency(self._h, out.ctypes.data_as(_ip), out.size):
            raise RuntimeError("get_adjacency failed")
        return out

    def stats(self) -> dict:
        s = Stats()
        if self._L.pumitally_get_stats(self._h, C.byref(s)):
            raise RuntimeError("get_stats failed")
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    def debug_order(self):
        out = np.empty(self.num_particles, dtype=np.int32)
        cnt = int(self._L.pumitally_debug_order(self._h, out.ctypes.data_as(_ip), out.size))
        return out[:max(cnt, 0)]

    def reset_tally(self):
        self._L.pumitally_reset_tally(self._h)

    def set_source_normalization(self, mode: int, value: float = 1.0):
        """0 volume only (reference), 1 /num_particles, 2 /value, 3 /total weight of the batch's first tracks."""
        if self._L.pumitally_set_source_normalization(self._h, int(mode), float(value)):
            raise ValueError(f"bad source normalisation mode={mode} value={value}")

    def source_normalization(self) -> float:
        return float(self._L.pumitally_get_source_normalization(self._h))

    # ---- batch statistics --------------------------------------------------------
    def end_batch(self):
        """Close the batch: its normalised tally joins the running sums, the tally starts over (collective)."""
        if self._L.pumitally_end_batch(self._h):
            raise RuntimeError("end_batch failed")

    def tally_statistics(self):
        """(mean, std_dev) over the ended batches, per unit volume: shape (E,), or (nbins, E) with score bins."""
        nb = self.score_bins
        shape = (self.num_elements,) if nb == 1 else (nb, self.num_elements)
        mean, std = np.empty(shape), np.empty(shape)
        if self._L.pumitally_get_tally_statistics(self._h, mean.ctypes.data_as(_dp), std.ctypes.data_as(_dp), mean.size):
            raise RuntimeError("get_tally_statistics failed")
        return mean, std

    def max_relative_error(self, threshold: float):
        """(max std_dev/|mean|, bin * E + element id where it is reached, pairs above threshold); n >= 2."""
        r, i, c = C.c_double(), C.c_int64(), C.c_int64()
        if self._L.pumitally_get_max_relative_error(self._h, float(threshold), C.byref(r), C.byref(i), C.byref(c)):
            raise RuntimeError("get_max_relative_error failed")
        return r.value, i.value, c.value

    def set_option(self, name: str, value: int):
        if self._L.pumitally_set_option(self._h, name.encode(), int(value)):
            raise ValueError(f"bad option {name}={value}")

    def get_option(self, name: str) -> int:
        return int(self._L.pumitally_get_option(self._h, name.encode()))

    # ---- multi-GPU -------------------------------------------------------------
    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = (C.c_uint8 * 128)()
        if load_library().pumitally_nccl_unique_id(buf):
            raise RuntimeError("ncclGetUniqueId failed")
        return bytes(buf)

    def comm_init(self, rank: int, nranks: int, unique_id: bytes):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        if self._L.pumitally_comm_init(self._h, rank, nranks, buf):
            raise RuntimeError("ncclCommInitRank failed")

    def allreduce_tally(self):
        if self._L.pumitally_allreduce_tally(self._h):
            raise RuntimeError("allreduce_tally failed")

    def exchange_tally(self):
        """Batch-end exchange: the quicker of the two below on this mesh, as measured by comm_init."""
        if self._L.pumitally_exchange_tally(self._h):
            raise RuntimeError("exchange_tally failed")

    def reduce_tally_to_owners(self):
        """Batch-end exchange by ncclReduceScatter; the flux accessors gather the shares (collective)."""
        if self._L.pumitally_reduce_tally_to_owners(self._h):
            raise RuntimeError("reduce_tally_to_owners failed")
