"""ctypes binding of libb200grav.so (include/b200grav.h) for the test and
benchmark harness.

The product is the C-ABI library; this module only marshals pointers.  Device
buffers are torch CUDA tensors (torch is plumbing: memory, streams,
torch.distributed) or raw integer device pointers.  There is no CPU fallback:
a missing library or a missing sm_100 GPU raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libb200grav.so")

EXPORTS = [
    "b200_error_string", "b200_abi_version", "b200_ctx_create", "b200_ctx_destroy",
    "b200_ctx_device", "b200_ctx_sm_count", "b200_ctx_stream", "b200_ctx_sync",
    "b200_direct_forces_host", "b200_direct_forces_dev", "b200_tiles_bytes",
    "b200_pack_tiles_dev", "b200_direct_forces_parts_dev",
    "b200_morton_keys_dev", "b200_sort_pairs_dev", "b200_tree_build_dev",
    "b200_tree_walk_dev", "b200_tree_forces_host", "b200_tree_stats", "b200_tree_export",
    "b200_tree_set_counting", "b200_tree_counters", "b200_tree_walk_stats", "b200_tree_overflowed",
    "b200_tree_build_part_dev", "b200_tree_forest_publish", "b200_tree_walk_list_dev", "b200_tree_forest_root",
    "b200_scatter_rows_dev", "b200_gather_rows_dev", "b200_host_register", "b200_host_unregister",
    "b200_leapfrog_dev", "b200_leapfrog_host", "b200_hubble_a", "b200_scale_factor_step", "b200_pack_posm_dev",
    "b200_device_alloc", "b200_device_free", "b200_memcpy_h2d", "b200_memcpy_d2h", "b200_unpack_pos3_dev", "b200_ipc_export", "b200_ipc_open", "b200_ipc_close",
    "b200_shard_range", "b200_shard_unique_id", "b200_shard_init", "b200_shard_finalize", "b200_shard_info",
    "b200_allgather_sources_dev", "b200_allreduce_sum_f64", "b200_direct_potential_dev", "b200_energy_dev",
    "b200_ic_params_default", "b200_zeldovich_ics_dev", "b200_force_error_dev", "b200_power_spectrum_dev", "b200_tree_build_fixed_dev", "b200_tree_forces_fixed_host", "b200_tree_set_periodic", "b200_spatial_order_dev", "b200_tree_build_host", "b200_tree_walk_host", "b200_tree_potential_dev", "b200_tree_energy_dev",
    "b200_fp32_peak_probe", "b200_last_kernel_ms", "b200_set_timing", "b200_launch_count",
    "b200_pm_forces_dev", "b200_pm_forces_host", "b200_pm_phase_ms",
]


class ICParams(C.Structure):
    """b200_ic_params (include/b200grav.h)."""
    _fields_ = [("grid", C.c_int), ("box", C.c_float), ("z_initial", C.c_double), ("seed", C.c_uint32),
                ("omega_m", C.c_double), ("omega_lambda", C.c_double), ("omega_k", C.c_double), ("h", C.c_double),
                ("sigma_8", C.c_double), ("n_s", C.c_double), ("particle_mass", C.c_float),
                ("origin_shift", C.c_float), ("use_2lpt", C.c_int)]


class B200Error(RuntimeError):
    pass


def load_library(path=None):
    path = path or os.environ.get("B200GRAV_LIB") or LIB_PATH      # B200GRAV_LIB: tuning hook (variant builds)
    if not os.path.exists(path):
        raise B200Error(
            f"{path} is missing: build it with `make -C lambda-cdm-raytracing_b200/csrc` "
            "(__graft_entry__.build()). There is no CPU fallback.")
    L = C.CDLL(path)
    sz, vp, f32, i32, f64 = C.c_size_t, C.c_void_p, C.c_float, C.c_int, C.c_double
    L.b200_error_string.restype = C.c_char_p
    L.b200_error_string.argtypes = [i32]
    L.b200_ctx_create.argtypes = [i32, sz, C.POINTER(vp)]
    L.b200_ctx_destroy.argtypes = [vp]
    L.b200_ctx_device.argtypes = [vp]
    L.b200_ctx_sm_count.argtypes = [vp]
    L.b200_ctx_sync.argtypes = [vp, vp]
    L.b200_ctx_stream.argtypes = [vp]
    L.b200_ctx_stream.restype = vp
    L.b200_direct_forces_host.argtypes = [vp, vp, vp, vp, sz, f32, f32]
    L.b200_direct_forces_dev.argtypes = [vp, vp, sz, sz, sz, f32, f32, vp, vp]
    L.b200_tiles_bytes.argtypes = [sz]
    L.b200_tiles_bytes.restype = sz
    L.b200_pack_tiles_dev.argtypes = [vp, vp, sz, vp, vp]
    L.b200_direct_forces_parts_dev.argtypes = [vp, C.POINTER(vp), C.POINTER(sz), i32, vp, sz, f32, f32, i32, vp, vp]
    L.b200_morton_keys_dev.argtypes = [vp, vp, sz, f32, vp, vp]
    L.b200_sort_pairs_dev.argtypes = [vp, vp, sz, vp, vp, vp]
    L.b200_tree_build_dev.argtypes = [vp, vp, sz, f32, i32, i32, vp]
    L.b200_tree_build_fixed_dev.argtypes = [vp, vp, sz, i32, i32, f32, vp]
    L.b200_tree_forces_fixed_host.argtypes = [vp, vp, vp, vp, sz, f32, i32, i32, f32]
    L.b200_tree_set_periodic.argtypes = [vp, f32]
    L.b200_spatial_order_dev.argtypes = [vp, vp, sz, f32, vp, vp]
    L.b200_tree_build_host.argtypes = [vp, vp, vp, sz, f32, i32, i32]
    L.b200_tree_walk_host.argtypes = [vp, vp, sz, f32]
    L.b200_tree_potential_dev.argtypes = [vp, sz, sz, f32, vp, vp]
    L.b200_tree_energy_dev.argtypes = [vp, sz, sz, vp, f32, C.POINTER(f64), C.POINTER(f64), vp]
    L.b200_tree_walk_dev.argtypes = [vp, sz, sz, f32, vp, vp]
    L.b200_tree_forces_host.argtypes = [vp, vp, vp, vp, sz, f32, i32, i32, f32]
    L.b200_tree_stats.argtypes = [vp] + [C.POINTER(sz)] * 4
    L.b200_tree_export.argtypes = [vp] + [vp] * 9
    L.b200_tree_set_counting.argtypes = [vp, i32]
    L.b200_tree_counters.argtypes = [vp, vp]
    L.b200_tree_walk_stats.argtypes = [vp, vp]
    L.b200_tree_overflowed.argtypes = [vp, C.POINTER(i32)]
    L.b200_tree_build_part_dev.argtypes = [vp, vp, vp, sz, f32, i32, i32, i32, i32, vp]
    L.b200_tree_forest_publish.argtypes = [vp, vp]
    L.b200_tree_walk_list_dev.argtypes = [vp, vp, sz, f32, vp, vp]
    L.b200_tree_forest_root.argtypes = [vp, vp]
    L.b200_scatter_rows_dev.argtypes = [vp, vp, vp, sz, vp, vp]
    L.b200_gather_rows_dev.argtypes = [vp, vp, vp, vp, sz, vp, vp, vp]
    L.b200_host_register.argtypes = [vp, vp, sz]
    L.b200_host_unregister.argtypes = [vp, vp]
    L.b200_leapfrog_dev.argtypes = [vp, vp, vp, vp, sz, i32, f32, f64, f32, f32, vp]
    L.b200_leapfrog_host.argtypes = [vp, vp, vp, vp, vp, sz, i32, f32, f64, f32, f32]
    L.b200_hubble_a.argtypes = [f64] * 5
    L.b200_hubble_a.restype = f64
    L.b200_scale_factor_step.argtypes = [f64] * 6
    L.b200_scale_factor_step.restype = f64
    L.b200_pack_posm_dev.argtypes = [vp, vp, vp, sz, vp, vp]
    L.b200_device_alloc.argtypes = [vp, sz, C.POINTER(vp)]
    L.b200_device_free.argtypes = [vp, vp]
    L.b200_memcpy_h2d.argtypes = [vp, vp, vp, sz, vp]
    L.b200_memcpy_d2h.argtypes = [vp, vp, vp, sz, vp]
    L.b200_unpack_pos3_dev.argtypes = [vp, vp, sz, vp, vp]
    L.b200_ipc_export.argtypes = [vp, vp, vp]
    L.b200_ipc_open.argtypes = [vp, vp, C.POINTER(vp)]
    L.b200_ipc_close.argtypes = [vp, vp]
    L.b200_shard_range.argtypes = [sz, i32, i32, C.POINTER(sz), C.POINTER(sz)]
    L.b200_shard_unique_id.argtypes = [vp]
    L.b200_shard_init.argtypes = [vp, vp, i32, i32]
    L.b200_shard_finalize.argtypes = [vp]
    L.b200_shard_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.b200_allgather_sources_dev.argtypes = [vp, vp, sz, vp]
    L.b200_allreduce_sum_f64.argtypes = [vp, vp, sz]
    L.b200_direct_potential_dev.argtypes = [vp, vp, sz, sz, sz, f32, f32, vp, vp]
    L.b200_energy_dev.argtypes = [vp, vp, sz, sz, sz, vp, f32, f32, C.POINTER(f64), C.POINTER(f64), vp]
    L.b200_ic_params_default.argtypes = [C.POINTER(ICParams)]
    L.b200_ic_params_default.restype = None
    L.b200_zeldovich_ics_dev.argtypes = [vp, C.POINTER(ICParams), sz, vp, vp, C.POINTER(f64), vp]
    L.b200_force_error_dev.argtypes = [vp, vp, vp, sz, C.POINTER(f64), C.POINTER(f64), vp]
    L.b200_power_spectrum_dev.argtypes = [vp, vp, sz, i32, f32, i32, i32, vp, vp, vp, vp]
    L.b200_pm_forces_dev.argtypes = [vp, vp, sz, sz, sz, i32, f32, f32, vp, vp, vp]
    L.b200_pm_forces_host.argtypes = [vp, vp, vp, vp, sz, i32, f32, f32]
    L.b200_pm_phase_ms.argtypes = [vp, vp]
    L.b200_fp32_peak_probe.argtypes = [vp, i32, i32, C.POINTER(f64), C.POINTER(f32)]
    L.b200_last_kernel_ms.argtypes = [vp, C.POINTER(f32)]
    L.b200_set_timing.argtypes = [vp, i32]
    L.b200_launch_count.argtypes = [vp]
    L.b200_launch_count.restype = C.c_uint64
    return L


def _ptr(x):
    """Device/host pointer of a torch tensor, numpy array, int or None."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    raise TypeError(type(x))


def _stream(stream):
    if stream is None:
        import torch
        return torch.cuda.current_stream().cuda_stream
    if isinstance(stream, int):
        return stream
    return stream.cuda_stream


class Engine:
    """One b200_ctx: the device-side state behind a force computer."""

    def __init__(self, device=0, max_particles=0, lib=None):
        self.L = lib or load_library()
        h = C.c_void_p()
        self._h = None
        self._check(self.L.b200_ctx_create(device, max_particles, C.byref(h)))
        self._h = h
        self.device = device

    def _check(self, rc):
        if rc != 0:
            raise B200Error(f"b200grav status {rc}: {self.L.b200_error_string(rc).decode()}")

    def close(self):
        if self._h is not None:
            self.L.b200_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def sm_count(self):
        return self.L.b200_ctx_sm_count(self._h)

    @property
    def launches(self):
        return int(self.L.b200_launch_count(self._h))

    def sync(self, stream=0):
        self._check(self.L.b200_ctx_sync(self._h, stream or None))

    # -- direct --------------------------------------------------------------
    def direct_forces_host(self, pos, mass=None, eps=0.01, box=0.0, out=None):
        pos = np.ascontiguousarray(pos, np.float32)
        n = pos.shape[0]
        m = None if mass is None else np.ascontiguousarray(mass, np.float32)
        if out is None:
            out = np.empty((n, 3), np.float32)
        self._check(self.L.b200_direct_forces_host(self._h, _ptr(pos), _ptr(m), _ptr(out), n, eps, box))
        return out

    def direct_forces_dev(self, posm, acc, i0=0, n_targets=None, eps=0.01, box=0.0, stream=None):
        n = posm.shape[0]
        nt = n - i0 if n_targets is None else n_targets
        self._check(self.L.b200_direct_forces_dev(self._h, _ptr(posm), n, i0, nt, eps, box, _ptr(acc),
                                                  _stream(stream)))
        return acc

    def tiles_bytes(self, n):
        return int(self.L.b200_tiles_bytes(n))

    def pack_tiles_dev(self, posm, n, tiles, stream=None):
        self._check(self.L.b200_pack_tiles_dev(self._h, _ptr(posm), n, _ptr(tiles), _stream(stream)))

    def direct_forces_parts_dev(self, parts, part_len, targets, n_targets, acc, eps=0.01, box=0.0, stream=None,
                                all_masses_equal=False):
        k = len(parts)
        arr_p = (C.c_void_p * k)(*[_ptr(p) for p in parts])
        arr_n = (C.c_size_t * k)(*part_len)
        self._check(self.L.b200_direct_forces_parts_dev(self._h, arr_p, arr_n, k, _ptr(targets), n_targets,
                                                        eps, box, int(all_masses_equal), _ptr(acc), _stream(stream)))
        return acc

    # -- tree ----------------------------------------------------------------
    def morton_keys_dev(self, posm, n, box, keys, stream=None):
        self._check(self.L.b200_morton_keys_dev(self._h, _ptr(posm), n, box, _ptr(keys), _stream(stream)))

    def sort_pairs_dev(self, keys_in, n, keys_out, perm_out, stream=None):
        self._check(self.L.b200_sort_pairs_dev(self._h, _ptr(keys_in), n, _ptr(keys_out), _ptr(perm_out),
                                               _stream(stream)))

    def tree_build_dev(self, posm, n, box=100.0, leaf_cap=8, max_depth=20, stream=None):
        self._check(self.L.b200_tree_build_dev(self._h, _ptr(posm), n, box, leaf_cap, max_depth, _stream(stream)))

    def tree_build_fixed_dev(self, posm, n, leaf_cap=8, max_depth=20, eps=0.01, stream=None):
        self._check(self.L.b200_tree_build_fixed_dev(self._h, _ptr(posm), n, leaf_cap, max_depth, eps, _stream(stream)))

    def tree_forces_fixed_host(self, pos, mass, theta=0.5, leaf_cap=8, max_depth=20, eps=0.01, out=None):
        pos = np.ascontiguousarray(pos, np.float32)
        mass = None if mass is None else np.ascontiguousarray(mass, np.float32)
        out = np.empty_like(pos) if out is None else out
        self._check(self.L.b200_tree_forces_fixed_host(self._h, _ptr(pos), _ptr(mass), _ptr(out), pos.shape[0],
                                                       theta, leaf_cap, max_depth, eps))
        return out

    def tree_potential_dev(self, phi, i0, n_targets, theta=0.5, stream=None):
        self._check(self.L.b200_tree_potential_dev(self._h, i0, n_targets, theta, _ptr(phi), _stream(stream)))

    def tree_energy_dev(self, vel, i0, n_targets, theta=0.5, stream=None):
        ke, pe = C.c_double(), C.c_double()
        self._check(self.L.b200_tree_energy_dev(self._h, i0, n_targets, _ptr(vel), theta, C.byref(ke), C.byref(pe),
                                                _stream(stream)))
        return ke.value, pe.value

    def spatial_order_dev(self, posm, n, box, perm, stream=None):
        """perm[k] = index of the k-th particle along a Hilbert curve over [-box/2, box/2)^3."""
        self._check(self.L.b200_spatial_order_dev(self._h, _ptr(posm), n, box, _ptr(perm), _stream(stream)))

    def tree_set_periodic(self, box):
        """Fixed-physics walks: minimum-image separations in a periodic box (0 = open boundary)."""
        self._check(self.L.b200_tree_set_periodic(self._h, box))

    def tree_walk_dev(self, acc, i0, n_targets, theta=0.5, stream=None):
        self._check(self.L.b200_tree_walk_dev(self._h, i0, n_targets, theta, _ptr(acc), _stream(stream)))
        return acc

    def tree_forces_host(self, pos, mass, theta=0.5, leaf_cap=8, max_depth=20, box=100.0, out=None):
        pos = np.ascontiguousarray(pos, np.float32)
        mass = np.ascontiguousarray(mass, np.float32)
        n = pos.shape[0]
        if out is None:
            out = np.empty((n, 3), np.float32)
        self._check(self.L.b200_tree_forces_host(self._h, _ptr(pos), _ptr(mass), _ptr(out), n, theta,
                                                 leaf_cap, max_depth, box))
        return out

    def tree_stats(self):
        v = [C.c_size_t() for _ in range(4)]
        self._check(self.L.b200_tree_stats(self._h, *[C.byref(x) for x in v]))
        return dict(n_nodes=v[0].value, n_leaves=v[1].value, depth=v[2].value, n_stored=v[3].value)

    def tree_export(self):
        st = self.tree_stats()
        nn, ns = st["n_nodes"], st["n_stored"]
        d = dict(level=np.empty(nn, np.int32), center=np.empty((nn, 3), np.float32),
                 size=np.empty(nn, np.float32), first_child=np.empty(nn, np.int32),
                 arrivals=np.empty(nn, np.int64), part_off=np.empty(nn + 1, np.int64),
                 part_idx=np.empty(max(ns, 1), np.int32), mass=np.empty(nn, np.float32),
                 com=np.empty((nn, 3), np.float32))
        self._check(self.L.b200_tree_export(self._h, *[_ptr(d[k]) for k in (
            "level", "center", "size", "first_child", "arrivals", "part_off", "part_idx", "mass", "com")]))
        d["part_idx"] = d["part_idx"][:ns]
        return d

    def tree_set_counting(self, on):
        self._check(self.L.b200_tree_set_counting(self._h, int(on)))

    def tree_counters(self):
        c = np.zeros(3, np.uint64)
        self._check(self.L.b200_tree_counters(self._h, _ptr(c)))
        return c

    # -- octant-sharded build / forest walk ------------------------------------
    def tree_build_part_dev(self, posm, n, part=0, n_parts=1, box=100.0, leaf_cap=8, max_depth=20, arrival=None,
                            stream=None):
        """Part `part` of an octant-sharded build (n_parts = 1: the whole tree); arrival: device int32[n], slot of
        the k-th particle in the reference's insertion order (None: stored in insertion order)."""
        self._check(self.L.b200_tree_build_part_dev(self._h, _ptr(posm), _ptr(arrival), n, box, leaf_cap, max_depth,
                                                    part, n_parts, _stream(stream)))

    def tree_forest_publish(self, stream=None):
        self._check(self.L.b200_tree_forest_publish(self._h, _stream(stream)))

    def tree_walk_list_dev(self, acc, target_list, n_list=None, theta=0.5, stream=None):
        n_list = target_list.shape[0] if n_list is None else n_list
        self._check(self.L.b200_tree_walk_list_dev(self._h, _ptr(target_list), n_list, theta, _ptr(acc),
                                                   _stream(stream)))
        return acc

    def tree_forest_root(self):
        out = np.zeros(8, np.float32)
        self._check(self.L.b200_tree_forest_root(self._h, _ptr(out)))
        return out

    def scatter_rows_dev(self, src4, perm, n, dst4, stream=None):
        self._check(self.L.b200_scatter_rows_dev(self._h, _ptr(src4), _ptr(perm), n, _ptr(dst4), _stream(stream)))

    def gather_rows_dev(self, src4, src3, index_list, n, out4, out3, stream=None):
        self._check(self.L.b200_gather_rows_dev(self._h, _ptr(src4), _ptr(src3), _ptr(index_list), n, _ptr(out4),
                                                _ptr(out3), _stream(stream)))

    def host_register(self, array):
        self._check(self.L.b200_host_register(self._h, _ptr(array), array.nbytes))

    def host_unregister(self, array):
        self._check(self.L.b200_host_unregister(self._h, _ptr(array)))

    def tree_walk_stats(self):
        """Counters of the last counting walk + lane utilisation: nodes visited, cell, pair interactions,
        pair-row source slots issued, node-visit lanes issued, node-visit lanes awake."""
        c = np.zeros(6, np.uint64)
        self._check(self.L.b200_tree_walk_stats(self._h, _ptr(c)))
        return c

    def tree_overflowed(self):
        f = C.c_int()
        self._check(self.L.b200_tree_overflowed(self._h, C.byref(f)))
        return bool(f.value)

    # -- leapfrog ------------------------------------------------------------
    def leapfrog_dev(self, posm, vel, acc, n, n_kicks, dt_kick, a, dt_drift, box, stream=None):
        self._check(self.L.b200_leapfrog_dev(self._h, _ptr(posm), _ptr(vel), _ptr(acc), n, n_kicks, dt_kick,
                                             a, dt_drift, box, _stream(stream)))

    def leapfrog_host(self, pos, vel, acc, mass, n_kicks, dt_kick, a, dt_drift, box):
        n = pos.shape[0]
        m = None if mass is None else np.ascontiguousarray(mass, np.float32)
        self._check(self.L.b200_leapfrog_host(self._h, _ptr(pos), _ptr(vel), _ptr(np.ascontiguousarray(acc, np.float32)),
                                              _ptr(m), n, n_kicks, dt_kick, a, dt_drift, box))

    def hubble_a(self, a, om=0.31, ok=0.0, ol=0.69, h=0.67):
        return float(self.L.b200_hubble_a(a, om, ok, ol, h))

    def scale_factor_step(self, a, dt, om=0.31, ok=0.0, ol=0.69, h=0.67):
        return float(self.L.b200_scale_factor_step(a, dt, om, ok, ol, h))

    def pack_posm_dev(self, pos3, mass, n, posm, stream=None):
        self._check(self.L.b200_pack_posm_dev(self._h, _ptr(pos3), _ptr(mass), n, _ptr(posm), _stream(stream)))

    # -- multi-GPU -----------------------------------------------------------
    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._check(self.L.b200_device_alloc(self._h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, ptr):
        self._check(self.L.b200_device_free(self._h, ptr))

    def ipc_export(self, tensor_or_ptr):
        h = (C.c_ubyte * 64)()
        self._check(self.L.b200_ipc_export(self._h, _ptr(tensor_or_ptr), C.addressof(h)))
        return bytes(h)

    def ipc_open(self, handle):
        buf = (C.c_ubyte * 64).from_buffer_copy(handle)
        p = C.c_void_p()
        self._check(self.L.b200_ipc_open(self._h, C.addressof(buf), C.byref(p)))
        return p.value

    def ipc_close(self, ptr):
        self._check(self.L.b200_ipc_close(self._h, ptr))

    # -- measurement ---------------------------------------------------------
    # ---- initial conditions ----
    def zeldovich_ics_dev(self, posm, vel, n_particles=None, stream=None, **params):
        """Fill posm float4[n] / vel float[3n] (device) with Zel'dovich particles; params override the
        reference's defaults (grid, box, z_initial, seed, omega_m, ..., particle_mass, origin_shift).
        Returns (rms displacement, largest displacement, growth factor, a*H*f)."""
        p = ICParams()
        self.L.b200_ic_params_default(C.byref(p))
        for k, v in params.items():
            if not hasattr(p, k):
                raise TypeError(f"unknown initial-conditions parameter {k!r}")
            setattr(p, k, v)
        n = p.grid ** 3 if n_particles is None else n_particles
        st = (C.c_double * 4)()
        self._check(self.L.b200_zeldovich_ics_dev(self._h, C.byref(p), n, _ptr(posm), _ptr(vel), st, _stream(stream)))
        return tuple(st)

    # ---- diagnostics ----
    def force_error_dev(self, acc_test, acc_ref, n=None, stream=None):
        """(mean, max) of |a_test - a_ref| / (|a_ref| + 1e-10) over the particles."""
        n = acc_ref.shape[0] if n is None else n
        a, m = C.c_double(), C.c_double()
        self._check(self.L.b200_force_error_dev(self._h, _ptr(acc_test), _ptr(acc_ref), n, C.byref(a), C.byref(m),
                                                _stream(stream)))
        return a.value, m.value

    def power_spectrum_dev(self, posm, grid, box, mass_weighted=True, shot_noise_correction=True, n=None, stream=None):
        """(k, P(k), modes per bin) of the particles: CIC mesh of grid^3, bins of width 2 pi / box."""
        n = posm.shape[0] if n is None else n
        nb = grid // 2
        k, p, c = np.empty(nb, np.float32), np.empty(nb, np.float32), np.empty(nb, np.int32)
        self._check(self.L.b200_power_spectrum_dev(self._h, _ptr(posm), n, grid, box, int(mass_weighted),
                                                   int(shot_noise_correction), _ptr(k), _ptr(p), _ptr(c), _stream(stream)))
        return k, p, c

    # ---- periodic particle mesh ----
    def pm_forces_dev(self, posm, acc, i0=0, n_targets=None, grid=128, box=100.0, r_split=None, phi=None,
                      stream=None):
        """Periodic long-range PM acceleration of targets posm[i0 : i0+n_targets) from all of posm (device);
        phi (device float[n_targets] or None): the positive long-range potential.  r_split=None: 1.25 box / grid."""
        n = posm.shape[0]
        nt = n - i0 if n_targets is None else n_targets
        rs = 1.25 * box / grid if r_split is None else r_split
        self._check(self.L.b200_pm_forces_dev(self._h, _ptr(posm), n, i0, nt, grid, box, rs, _ptr(acc), _ptr(phi),
                                              _stream(stream)))
        return acc

    def pm_forces_host(self, pos, mass, grid, box, r_split=None, out=None):
        pos = np.ascontiguousarray(pos, np.float32)
        n = pos.shape[0]
        m = None if mass is None else np.ascontiguousarray(mass, np.float32)
        if out is None:
            out = np.empty((n, 3), np.float32)
        rs = 1.25 * box / grid if r_split is None else r_split
        self._check(self.L.b200_pm_forces_host(self._h, _ptr(pos), _ptr(m), _ptr(out), n, grid, box, rs))
        return out

    def pm_phase_ms(self):
        """Phase times (ms) of the last timed pm_forces_dev: deposit, convert, R2C, k-space, C2R, interpolation,
        whole call."""
        ms = np.zeros(7, np.float32)
        self._check(self.L.b200_pm_phase_ms(self._h, _ptr(ms)))
        return ms

    # ---- energy diagnostic ----
    def direct_potential_dev(self, posm, phi, i0=0, n_targets=None, eps=0.01, box=0.0, stream=None):
        n = posm.shape[0]
        nt = n - i0 if n_targets is None else n_targets
        self._check(self.L.b200_direct_potential_dev(self._h, _ptr(posm), n, i0, nt, eps, box, _ptr(phi), _stream(stream)))

    def energy_dev(self, posm, vel, i0=0, n_targets=None, eps=0.01, box=0.0, stream=None):
        """(kinetic, potential) of targets [i0, i0+n_targets) as host floats; vel = their velocities."""
        n = posm.shape[0]
        nt = n - i0 if n_targets is None else n_targets
        ke, pe = C.c_double(), C.c_double()
        self._check(self.L.b200_energy_dev(self._h, _ptr(posm), n, i0, nt, _ptr(vel), eps, box,
                                           C.byref(ke), C.byref(pe), _stream(stream)))
        return ke.value, pe.value

    def allreduce_sum_f64(self, values):
        arr = np.ascontiguousarray(values, np.float64)
        self._check(self.L.b200_allreduce_sum_f64(self._h, arr.ctypes.data, arr.size))
        return arr

    # ---- NCCL source all-gather owned by the context (hosts without torch.distributed) ----
    def shard_unique_id(self):
        buf = (C.c_ubyte * 128)()
        self._check(self.L.b200_shard_unique_id(buf))
        return bytes(buf)

    def shard_init(self, unique_id, rank, world):
        buf = (C.c_ubyte * 128).from_buffer_copy(unique_id) if unique_id is not None else None
        self._check(self.L.b200_shard_init(self._h, buf, rank, world))

    def shard_finalize(self):
        self._check(self.L.b200_shard_finalize(self._h))

    def shard_info(self):
        r, w = C.c_int(), C.c_int()
        self._check(self.L.b200_shard_info(self._h, C.byref(r), C.byref(w)))
        return r.value, w.value

    def allgather_sources_dev(self, posm_full, n_total, stream=None):
        self._check(self.L.b200_allgather_sources_dev(self._h, _ptr(posm_full), n_total, _stream(stream)))

    def fp32_peak_probe(self, mode=0, iters=2000):
        t, ms = C.c_double(), C.c_float()
        self._check(self.L.b200_fp32_peak_probe(self._h, mode, iters, C.byref(t), C.byref(ms)))
        return t.value, ms.value

    def set_timing(self, on):
        self._check(self.L.b200_set_timing(self._h, int(on)))

    def last_kernel_ms(self):
        ms = C.c_float()
        self._check(self.L.b200_last_kernel_ms(self._h, C.byref(ms)))
        return ms.value


class LambdaCDMSimulation:
    """Device-resident KDK leapfrog driver with the call shape of the reference's
    physics::LambdaCDMSimulation (include/physics/lambda_cdm.hpp:22-75;
    step order src/physics/lambda_cdm_impl.cu:167-213), driving the C ABI.

    force: "direct", "tree" or "pm" (periodic particle mesh on a pm_grid^3 mesh, Gaussian split radius r_split,
    None = 1.25 box / pm_grid).  The first half-kick of the first step uses the
    forces at the initial positions (the reference reads uninitialised memory
    there; SURVEY 8c)."""

    def __init__(self, engine, pos, vel, mass, box=100.0, force="direct", eps=0.01, theta=0.5,
                 leaf_cap=8, max_depth=20, wrap=True, a0=1.0, cosmo=(0.31, 0.0, 0.69, 0.67),
                 i0=0, n_local=None, gather=None, pm_grid=128, r_split=None):
        import torch
        self.torch = torch
        self.e = engine
        dev = torch.device("cuda", engine.device)
        n = pos.shape[0]
        self.n = n
        self.i0 = i0
        self.nl = n - i0 if n_local is None else n_local
        self.box, self.force, self.eps, self.theta = float(box), force, float(eps), float(theta)
        self.leaf_cap, self.max_depth, self.wrap = leaf_cap, max_depth, wrap
        self.a = float(a0)
        self.cosmo = cosmo
        self.gather = gather              # callable(posm_full) -> refreshes non-local rows (multi-GPU)
        self.pm_grid = int(pm_grid)
        self.r_split = 1.25 * self.box / self.pm_grid if r_split is None else float(r_split)
        pm = np.concatenate([np.asarray(pos, np.float32), np.asarray(mass, np.float32)[:, None]], axis=1)
        self.posm = torch.from_numpy(np.ascontiguousarray(pm)).to(dev)
        self.vel = torch.from_numpy(np.ascontiguousarray(vel, np.float32)[i0:i0 + self.nl].copy()).to(dev)
        self.acc = torch.zeros((self.nl, 3), dtype=torch.float32, device=dev)
        self.steps = 0
        self.have_forces = False

    def compute_forces(self):
        if self.force == "direct":
            self.e.direct_forces_dev(self.posm, self.acc, self.i0, self.nl, self.eps, 0.0)
        elif self.force == "pm":
            self.e.pm_forces_dev(self.posm, self.acc, self.i0, self.nl, self.pm_grid, self.box, self.r_split)
        else:
            self.e.tree_build_dev(self.posm, self.n, self.box, self.leaf_cap, self.max_depth)
            self.e.tree_walk_dev(self.acc, self.i0, self.nl, self.theta)
        self.have_forces = True

    def step(self, dt):
        e = self.e
        if not self.have_forces:
            self.compute_forces()
        local = self.posm[self.i0:self.i0 + self.nl]
        wrap_box = self.box if self.wrap else 0.0
        # opening half-kick + drift (fused)
        e.leapfrog_dev(local, self.vel, self.acc, self.nl, 1, np.float32(dt * 0.5), self.a, np.float32(dt), wrap_box)
        self.a = e.scale_factor_step(self.a, dt, *self.cosmo)
        if self.gather is not None:
            self.gather(self.posm)
        self.compute_forces()
        # closing half-kick with the new scale factor
        e.leapfrog_dev(local, self.vel, self.acc, self.nl, 1, np.float32(dt * 0.5), self.a, 0.0, wrap_box)
        self.steps += 1

    def get_scale_factor(self):
        return self.a

    def positions(self):
        return self.posm[:, :3].cpu().numpy()

    def velocities(self):
        return self.vel.cpu().numpy()


# ---------------------------------------------------------------------------
# Target-sharded data parallelism (SURVEY 8e): rank r owns the contiguous
# original-index range [r*N/G, (r+1)*N/G) of the targets; sources are all-gathered.
def shard_range(n, rank, world):
    return rank * n // world, (rank + 1) * n // world


class SourceGather:
    """All-gathers each rank's float4 shard into the replicated posm array with
    torch.distributed (NCCL on GPUs, gloo in the CPU tests).  Semantic ancestor:
    ClusterCommunicator::gather_all_particles (reference src/mpi/cluster_comm.cpp:218-247)."""

    def __init__(self, n, rank, world, group=None):
        self.n, self.rank, self.world, self.group = n, rank, world, group
        self.lo, self.hi = shard_range(n, rank, world)
        self.equal = (n % world == 0)

    def __call__(self, posm):
        import torch.distributed as dist
        if self.world == 1:
            return posm
        mine = posm[self.lo:self.hi].clone()
        if self.equal:
            dist.all_gather_into_tensor(posm.view(-1), mine.view(-1), group=self.group)
        else:
            outs = [posm[slice(*shard_range(self.n, r, self.world))] for r in range(self.world)]
            if posm.is_cuda:
                dist.all_gather(outs, mine, group=self.group)
            else:   # gloo needs equal-sized outputs: pad
                width = max(o.shape[0] for o in outs)
                import torch
                pad = torch.zeros((width, posm.shape[1]), dtype=posm.dtype)
                pad[: mine.shape[0]] = mine
                bufs = [torch.empty_like(pad) for _ in range(self.world)]
                dist.all_gather(bufs, pad, group=self.group)
                for o, b in zip(outs, bufs):
                    o.copy_(b[: o.shape[0]])
        return posm


class PeerSources:
    """The fused alternative to SourceGather for the direct sum: every rank packs its
    shard into a tile-SoA buffer it owns and exports (CUDA IPC); peers map it, and
    b200_direct_forces_parts_dev pulls source tiles straight out of peer HBM over
    NVLink with TMA bulk copies -- no all-gather, one barrier per step.
    Two buffers alternate so that a rank may repack while slower peers still read."""

    def __init__(self, engine, n, rank, world, barrier, exchange):
        self.e, self.n, self.rank, self.world, self.barrier = engine, n, rank, world, barrier
        self.lens = [shard_range(n, r, world)[1] - shard_range(n, r, world)[0] for r in range(world)]
        nbytes = max(engine.tiles_bytes(max(self.lens)), 8192)
        self.mine = [engine.device_alloc(nbytes) for _ in range(2)]
        handles = exchange([engine.ipc_export(p) for p in self.mine])       # list over ranks of [h0, h1]
        self.parts = [[self.mine[b] if r == rank else engine.ipc_open(handles[r][b]) for r in range(world)]
                      for b in range(2)]
        self.step = 0

    def publish(self, shard_posm, stream=None):
        """Pack this rank's float4 shard into the current buffer, then barrier."""
        b = self.step & 1
        self.e.pack_tiles_dev(shard_posm, self.lens[self.rank], self.mine[b], stream)
        self.barrier()
        self.step += 1
        return self.parts[b]

    def close(self):
        for b in range(2):
            for r in range(self.world):
                if r != self.rank:
                    self.e.ipc_close(self.parts[b][r])
            self.e.device_free(self.mine[b])
