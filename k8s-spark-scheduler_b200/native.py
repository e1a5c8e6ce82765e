"""ctypes binding of libgangpack.so (include/gangpack.h) -- the only compute path of this package.

There is deliberately no CPU fallback here: if the shared library is missing or no sm_100 device is
usable, loading / context creation raises.
"""
from __future__ import annotations

import ctypes as C
import glob
import os
import shutil
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
LIB_PATH = os.environ.get("GANGPACK_LIB") or os.path.join(_PKG, "libgangpack.so")   # GANGPACK_LIB: experimental builds
# every file the library is built from: an edit to any of them makes build() recompile
_SOURCES = sorted(glob.glob(os.path.join(_PKG, "csrc", "*.cu")) + glob.glob(os.path.join(_PKG, "csrc", "*.cuh"))) + [
    os.path.join(_ROOT, "include", "gangpack.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]

TIGHTLY_PACK = 0
DISTRIBUTE_EVENLY = 1
MINIMAL_FRAGMENTATION = 2   # GP_MODE_INDEPENDENT only
MODE_INDEPENDENT = 0
MODE_FIFO_REFERENCE = 1
MODE_FIFO_EXACT = 2

STATUS_NAMES = {0: "GP_OK", 1: "GP_ERR_INVALID", 2: "GP_ERR_CUDA", 3: "GP_ERR_NO_DEVICE", 4: "GP_ERR_NO_SNAPSHOT",
                5: "GP_ERR_CAPACITY", 6: "GP_ERR_UNREPRESENTABLE"}

# every symbol include/gangpack.h declares (tests assert the .so exports exactly these)
EXPORTS = ["gp_abi_version", "gp_create", "gp_destroy", "gp_last_error", "gp_backend", "gp_alloc_pinned",
           "gp_free_pinned", "gp_register_host", "gp_unregister_host", "gp_set_snapshot", "gp_get_snapshot", "gp_pack_batch", "gp_pack_batch_wire", "gp_pack_one", "gp_set_schedulable", "gp_pack_batch_zones", "gp_pack_fifo_zones", "gp_reserve_placements", "gp_apply_usage_delta",
           "gp_set_snapshot_device", "gp_pack_batch_device", "gp_stream", "gp_synchronize", "gp_last_stats",
           "gp_potential_nodes", "gp_build_availability", "gp_build_reschedule_availability", "gp_prepare_cluster", "gp_reschedule_executors",
           "gp_multi_create", "gp_multi_destroy", "gp_multi_last_error", "gp_multi_size", "gp_multi_ctx",
           "gp_multi_set_snapshot", "gp_multi_pack_batch", "gp_multi_get_snapshot", "gp_multi_group_owner"]


class GangpackError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build libgangpack.so")


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into k8s-spark-scheduler_b200/libgangpack.so (in-tree)."""
    stale = force or not os.path.exists(LIB_PATH) or any(
        os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in _SOURCES)
    if stale:
        cmd = [_nvcc()] + NVCC_FLAGS + ["-I", os.path.join(_ROOT, "include"), "-o", LIB_PATH,
                                        os.path.join(_PKG, "csrc", "gangpack_api.cu"), os.path.join(_PKG, "csrc", "gangpack_multi.cu")]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        subprocess.check_call(cmd)
    return LIB_PATH


class gp_config(C.Structure):
    _fields_ = [("device", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32 * 6)]


CFG_ASYNC_SNAPSHOT = 1


class gp_nodes(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("avail_cpu_milli", C.c_void_p), ("avail_mem_bytes", C.c_void_p),
                ("avail_gpu", C.c_void_p), ("n_groups", C.c_int32), ("exec_off", C.c_void_p),
                ("exec_order", C.c_void_p), ("drv_off", C.c_void_p), ("drv_order", C.c_void_p)]


class gp_apps(C.Structure):
    _fields_ = [("n_apps", C.c_int32), ("drv_cpu_milli", C.c_void_p), ("drv_mem_bytes", C.c_void_p),
                ("drv_gpu", C.c_void_p), ("exe_cpu_milli", C.c_void_p), ("exe_mem_bytes", C.c_void_p),
                ("exe_gpu", C.c_void_p), ("exe_count", C.c_void_p), ("group", C.c_void_p),
                ("skip_if_no_fit", C.c_void_p), ("exec_out_off", C.c_void_p)]


class gp_apps_wire(C.Structure):
    _fields_ = [("n_apps", C.c_int32), ("quantity_bits", C.c_int32), ("mem_shift", C.c_int32), ("reserved", C.c_int32),
                ("drv_cpu", C.c_void_p), ("drv_mem", C.c_void_p), ("drv_gpu", C.c_void_p),
                ("exe_cpu", C.c_void_p), ("exe_mem", C.c_void_p), ("exe_gpu", C.c_void_p),
                ("exe_count", C.c_void_p), ("group", C.c_void_p), ("skip_if_no_fit", C.c_void_p), ("exec_out_off", C.c_void_p)]


class gp_results_wire(C.Structure):
    _fields_ = [("driver_node", C.c_void_p), ("executor_nodes", C.c_void_p), ("executor_nodes_cap", C.c_int64),
                ("node_bits", C.c_int32), ("reserved", C.c_int32)]


class gp_zone_results(C.Structure):
    _fields_ = [("zone", C.c_void_p), ("driver_node", C.c_void_p), ("executor_nodes", C.c_void_p), ("executor_nodes_cap", C.c_int64),
                ("avg_efficiency", C.c_void_p)]


class gp_reservation_table(C.Structure):
    _fields_ = [("rows_cap", C.c_int64), ("app", C.c_void_p), ("slot", C.c_void_p), ("node", C.c_void_p), ("cpu_milli", C.c_void_p),
                ("mem_bytes", C.c_void_p), ("gpu", C.c_void_p), ("n_rows", C.c_int64)]


class gp_results(C.Structure):
    _fields_ = [("driver_node", C.c_void_p), ("executor_nodes", C.c_void_p), ("executor_nodes_cap", C.c_int64)]


class gp_sort_input(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("avail_cpu_milli", C.c_void_p), ("avail_mem_bytes", C.c_void_p),
                ("n_zones", C.c_int32), ("zone_id", C.c_void_p), ("name_rank", C.c_void_p),
                ("is_driver_candidate", C.c_void_p), ("unschedulable", C.c_void_p), ("ready", C.c_void_p),
                ("driver_label_rank", C.c_void_p), ("executor_label_rank", C.c_void_p),
                ("avail_gpu", C.c_void_p), ("undefined_ties", C.c_void_p)]


class gp_usage_input(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("alloc_cpu_milli", C.c_void_p), ("alloc_mem_bytes", C.c_void_p), ("alloc_gpu", C.c_void_p),
                ("overhead_cpu_milli", C.c_void_p), ("overhead_mem_bytes", C.c_void_p), ("overhead_gpu", C.c_void_p),
                ("n_reservations", C.c_int64), ("res_node", C.c_void_p), ("res_cpu_milli", C.c_void_p),
                ("res_mem_bytes", C.c_void_p), ("res_gpu", C.c_void_p)]


class gp_reschedule(C.Structure):
    _fields_ = [("n_execs", C.c_int32), ("exe_cpu_milli", C.c_void_p), ("exe_mem_bytes", C.c_void_p), ("exe_gpu", C.c_void_p),
                ("group", C.c_void_p), ("min_frag", C.c_int32), ("reserved_cpu_milli", C.c_void_p),
                ("reserved_mem_bytes", C.c_void_p), ("reserved_gpu", C.c_void_p), ("host_off", C.c_void_p),
                ("host_nodes", C.c_void_p)]


class gp_stats(C.Structure):
    _fields_ = [("nodes_scanned", C.c_int64), ("drivers_tried", C.c_int64), ("kernel_launches", C.c_int64),
                ("pack_kernel_ns", C.c_int64), ("prep_kernel_ns", C.c_int64), ("scan_path_apps", C.c_int64),
                ("scan_path_nodes", C.c_int64), ("reserved", C.c_int64 * 1)]


_lib = None


def load():
    """dlopen libgangpack.so; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(this package has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.gp_abi_version.restype = C.c_int
    L.gp_create.restype = C.c_int
    L.gp_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(gp_config)]
    L.gp_destroy.restype = None
    L.gp_destroy.argtypes = [C.c_void_p]
    L.gp_last_error.restype = C.c_char_p
    L.gp_last_error.argtypes = [C.c_void_p]
    L.gp_backend.restype = C.c_int
    L.gp_backend.argtypes = [C.c_void_p]
    L.gp_alloc_pinned.restype = C.c_int
    L.gp_alloc_pinned.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.gp_free_pinned.restype = C.c_int
    L.gp_free_pinned.argtypes = [C.c_void_p, C.c_void_p]
    L.gp_register_host.restype = C.c_int
    L.gp_register_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.gp_unregister_host.restype = C.c_int
    L.gp_unregister_host.argtypes = [C.c_void_p, C.c_void_p]
    L.gp_set_snapshot.restype = C.c_int
    L.gp_set_snapshot.argtypes = [C.c_void_p, C.POINTER(gp_nodes)]
    L.gp_get_snapshot.restype = C.c_int
    L.gp_get_snapshot.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gp_pack_batch.restype = C.c_int
    L.gp_pack_batch.argtypes = [C.c_void_p, C.POINTER(gp_apps), C.c_int, C.c_int, C.POINTER(gp_results)]
    L.gp_pack_batch_wire.restype = C.c_int
    L.gp_pack_batch_wire.argtypes = [C.c_void_p, C.POINTER(gp_apps_wire), C.c_int, C.c_int, C.POINTER(gp_results_wire)]
    L.gp_set_schedulable.restype = C.c_int
    L.gp_set_schedulable.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gp_pack_batch_zones.restype = C.c_int
    L.gp_pack_batch_zones.argtypes = [C.c_void_p, C.POINTER(gp_apps), C.c_int, C.POINTER(gp_zone_results)]
    L.gp_pack_fifo_zones.restype = C.c_int
    L.gp_pack_fifo_zones.argtypes = [C.c_void_p, C.POINTER(gp_apps), C.c_int, C.c_int, C.POINTER(gp_zone_results)]
    L.gp_reserve_placements.restype = C.c_int
    L.gp_reserve_placements.argtypes = [C.c_void_p, C.POINTER(gp_apps), C.POINTER(gp_results), C.c_int32, C.POINTER(gp_reservation_table)]
    L.gp_apply_usage_delta.restype = C.c_int
    L.gp_apply_usage_delta.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
    L.gp_pack_one.restype = C.c_int
    L.gp_pack_one.argtypes = [C.c_void_p, C.c_int] + [C.c_int64] * 6 + [C.c_int32, C.POINTER(C.c_int32),
                                                                          C.POINTER(C.c_int32), C.c_void_p]
    L.gp_set_snapshot_device.restype = C.c_int
    L.gp_set_snapshot_device.argtypes = [C.c_void_p, C.POINTER(gp_nodes), C.c_int32, C.c_int32, C.c_void_p]
    L.gp_pack_batch_device.restype = C.c_int
    L.gp_pack_batch_device.argtypes = [C.c_void_p, C.POINTER(gp_apps), C.c_int, C.c_int, C.POINTER(gp_results), C.c_void_p]
    L.gp_stream.restype = C.c_void_p
    L.gp_stream.argtypes = [C.c_void_p]
    L.gp_synchronize.restype = C.c_int
    L.gp_synchronize.argtypes = [C.c_void_p]
    L.gp_last_stats.restype = C.c_int
    L.gp_last_stats.argtypes = [C.c_void_p, C.POINTER(gp_stats)]
    L.gp_build_availability.restype = C.c_int
    L.gp_build_availability.argtypes = [C.c_void_p, C.POINTER(gp_usage_input)] + [C.c_void_p] * 6
    L.gp_build_reschedule_availability.restype = C.c_int
    L.gp_build_reschedule_availability.argtypes = [C.c_void_p, C.POINTER(gp_usage_input)] + [C.c_void_p] * 3
    L.gp_prepare_cluster.restype = C.c_int
    L.gp_prepare_cluster.argtypes = [C.c_void_p, C.POINTER(gp_usage_input), C.POINTER(gp_sort_input), C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32)]
    L.gp_potential_nodes.restype = C.c_int
    L.gp_potential_nodes.argtypes = [C.c_void_p, C.POINTER(gp_sort_input), C.c_void_p, C.POINTER(C.c_int32),
                                     C.c_void_p, C.POINTER(C.c_int32)]
    L.gp_reschedule_executors.restype = C.c_int
    L.gp_reschedule_executors.argtypes = [C.c_void_p, C.POINTER(gp_reschedule), C.c_void_p]
    L.gp_multi_create.restype = C.c_int
    L.gp_multi_create.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.c_int32]
    L.gp_multi_destroy.restype = None
    L.gp_multi_destroy.argtypes = [C.c_void_p]
    L.gp_multi_last_error.restype = C.c_char_p
    L.gp_multi_last_error.argtypes = [C.c_void_p]
    L.gp_multi_size.restype = C.c_int32
    L.gp_multi_size.argtypes = [C.c_void_p]
    L.gp_multi_ctx.restype = C.c_void_p
    L.gp_multi_ctx.argtypes = [C.c_void_p, C.c_int32]
    L.gp_multi_set_snapshot.restype = C.c_int
    L.gp_multi_set_snapshot.argtypes = [C.c_void_p, C.POINTER(gp_nodes)]
    L.gp_multi_pack_batch.restype = C.c_int
    L.gp_multi_pack_batch.argtypes = [C.c_void_p, C.POINTER(gp_apps_wire), C.c_int, C.c_int, C.POINTER(gp_results_wire)]
    L.gp_multi_get_snapshot.restype = C.c_int
    L.gp_multi_get_snapshot.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gp_multi_group_owner.restype = C.c_int
    L.gp_multi_group_owner.argtypes = [C.c_void_p, C.c_void_p]
    _lib = L
    return L


def _np(a, dtype):
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


def _p(a):
    return None if a is None else a.ctypes.data


def compact_apps(apps: dict, mem_shift: int = 20):
    """What the shim does while marshalling: the 32-bit wire layout when every quantity is exactly representable
    (memory a whole multiple of 2^mem_shift bytes, everything < 2^31), else None (use the int64 layout)."""
    out = dict(apps)
    for k in ("drv_cpu", "drv_gpu", "exe_cpu", "exe_gpu", "drv_mem", "exe_mem"):
        v = apps.get(k)
        if v is None:
            continue
        v = np.asarray(v, np.int64)
        if k.endswith("mem"):
            if (v & ((1 << mem_shift) - 1)).any():
                return None
            v = v >> mem_shift
        if (v < 0).any() or (v >= (1 << 31)).any():
            return None
        out[k] = v.astype(np.int32)
    return out


class PinnedArray:
    """numpy view over gp_alloc_pinned memory."""

    def __init__(self, packer: "GangPacker", shape, dtype):
        self._packer = packer
        self.dtype = np.dtype(dtype)
        n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
        self.nbytes = max(n * self.dtype.itemsize, 1)
        ptr = C.c_void_p()
        packer._check(load().gp_alloc_pinned(packer._h, self.nbytes, C.byref(ptr)))
        self._ptr = ptr
        buf = (C.c_char * self.nbytes).from_address(ptr.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=n).reshape(shape)

    def free(self):
        if self._ptr is not None and self._packer._h:
            self.array = None
            load().gp_free_pinned(self._packer._h, self._ptr)
            self._ptr = None


class GangPacker:
    """One gp_ctx.  Not thread-safe (like the C ABI)."""

    def __init__(self, device: int = -1, async_snapshot: bool = False):
        L = load()
        self._h = C.c_void_p()
        cfg = gp_config(device=device, flags=CFG_ASYNC_SNAPSHOT if async_snapshot else 0)
        st = L.gp_create(C.byref(self._h), C.byref(cfg))
        if st != 0:
            raise GangpackError(st, (L.gp_last_error(None) or b"").decode())
        self._keep = None
        self._pinned = []
        self._registered = []

    def close(self):
        if getattr(self, "_h", None):
            for p in self._pinned:
                p.free()
            self._pinned = []
            for addr in self._registered:
                load().gp_unregister_host(self._h, addr)
            self._registered = []
            load().gp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st: int):
        if st != 0:
            raise GangpackError(st, (load().gp_last_error(self._h) or b"").decode())

    def pinned(self, shape, dtype) -> np.ndarray:
        p = PinnedArray(self, shape, dtype)
        self._pinned.append(p)
        return p.array

    def register_host(self, array: np.ndarray):
        """Page-lock caller-owned memory (e.g. a shared-memory segment) so results can be DMA'd straight into it."""
        self._check(load().gp_register_host(self._h, array.ctypes.data, array.nbytes))
        self._registered.append(array.ctypes.data)

    def unregister_host(self, array: np.ndarray):
        self._check(load().gp_unregister_host(self._h, array.ctypes.data))
        self._registered.remove(array.ctypes.data)

    def pinned_columns(self, n: int, names, dtype=np.int64) -> dict:
        """`names` equally spaced columns of n elements inside ONE pinned block (column after column): the layout
        that lets gp_pack_batch move all int64 columns of a chunk with a single 2-D DMA."""
        block = self.pinned((len(names), n), dtype)
        return {name: block[i] for i, name in enumerate(names)}

    # ---- snapshot ----------------------------------------------------------------------------
    def set_snapshot(self, avail_cpu, avail_mem, avail_gpu, exec_order, drv_order, exec_off=None, drv_off=None):
        cpu, mem = _np(avail_cpu, np.int64), _np(avail_mem, np.int64)
        gpu = _np(avail_gpu, np.int64)
        eo, do = _np(exec_order, np.int32), _np(drv_order, np.int32)
        eoff = _np(exec_off if exec_off is not None else [0, len(eo)], np.int32)
        doff = _np(drv_off if drv_off is not None else [0, len(do)], np.int32)
        n = gp_nodes(n_nodes=len(cpu), avail_cpu_milli=_p(cpu), avail_mem_bytes=_p(mem), avail_gpu=_p(gpu),
                     n_groups=len(eoff) - 1, exec_off=_p(eoff), exec_order=_p(eo), drv_off=_p(doff), drv_order=_p(do))
        self._check(load().gp_set_snapshot(self._h, C.byref(n)))
        self.n_nodes = len(cpu)

    def get_snapshot(self):
        cpu = np.empty(self.n_nodes, np.int64); mem = np.empty(self.n_nodes, np.int64); gpu = np.empty(self.n_nodes, np.int64)
        self._check(load().gp_get_snapshot(self._h, _p(cpu), _p(mem), _p(gpu)))
        return cpu, mem, gpu

    # ---- executors without a usable reservation (rescheduleExecutor's node choice) -----------------
    def reschedule_executors(self, exe, min_frag=False, group=None, reserved=None, hosting=None):
        """exe: (cpu[q], mem[q], gpu[q]|None); reserved: (cpu[n], mem[n], gpu[n]|None) or None; hosting: list of
        per-executor node-index lists (nodes already hosting executors of the same application) or None.
        -> node index per executor (-1: no capacity)."""
        ec, em = _np(exe[0], np.int64), _np(exe[1], np.int64)
        eg = _np(exe[2], np.int64) if len(exe) > 2 else None
        q = len(ec)
        grp = _np(group, np.int32)
        rs = [_np(x, np.int64) for x in reserved] if reserved is not None else [None] * 3
        hoff = hn = None
        if hosting is not None:
            hoff = np.zeros(q + 1, np.int64)
            np.cumsum([len(h) for h in hosting], out=hoff[1:])
            hn = np.array([n for h in hosting for n in h] or [0], np.int32)
        out = np.full(max(q, 1), -9, np.int32)
        r = gp_reschedule(n_execs=q, exe_cpu_milli=_p(ec), exe_mem_bytes=_p(em), exe_gpu=_p(eg), group=_p(grp),
                          min_frag=1 if min_frag else 0, reserved_cpu_milli=_p(rs[0]), reserved_mem_bytes=_p(rs[1]),
                          reserved_gpu=_p(rs[2] if len(rs) > 2 else None), host_off=_p(hoff), host_nodes=_p(hn))
        self._check(load().gp_reschedule_executors(self._h, C.byref(r), _p(out)))
        return out[:q]

    # ---- availability snapshot from reservations (NodeSchedulingMetadataForNodes) ----------------
    def build_availability(self, alloc, overhead, res_node, res):
        """alloc / overhead / res: (cpu, mem, gpu) triples (overhead may be None) -> (avail triple, sched triple)."""
        al = [_np(x, np.int64) for x in alloc]
        ov = [_np(x, np.int64) for x in overhead] if overhead is not None else [None] * 3
        rn = _np(res_node, np.int32)
        rs = [_np(x, np.int64) for x in res]
        n = len(al[0])
        ui = gp_usage_input(n_nodes=n, alloc_cpu_milli=_p(al[0]), alloc_mem_bytes=_p(al[1]), alloc_gpu=_p(al[2]),
                            overhead_cpu_milli=_p(ov[0]), overhead_mem_bytes=_p(ov[1]), overhead_gpu=_p(ov[2]),
                            n_reservations=len(rn), res_node=_p(rn), res_cpu_milli=_p(rs[0]), res_mem_bytes=_p(rs[1]), res_gpu=_p(rs[2]))
        outs = [np.empty(max(n, 1), np.int64) for _ in range(6)]
        self._check(load().gp_build_availability(self._h, C.byref(ui), *[_p(o) for o in outs]))
        return [o[:n] for o in outs[:3]], [o[:n] for o in outs[3:]]

    def build_reschedule_availability(self, alloc, overhead, res_node, res):
        """availableResources of rescheduleExecutor's first-fit branch (overhead counted twice on nodes with reservations)."""
        al = [_np(x, np.int64) for x in alloc]
        ov = [_np(x, np.int64) for x in overhead] if overhead is not None else [None] * 3
        rn = _np(res_node, np.int32)
        rs = [_np(x, np.int64) for x in res]
        n = len(al[0])
        ui = gp_usage_input(n_nodes=n, alloc_cpu_milli=_p(al[0]), alloc_mem_bytes=_p(al[1]), alloc_gpu=_p(al[2]),
                            overhead_cpu_milli=_p(ov[0]), overhead_mem_bytes=_p(ov[1]), overhead_gpu=_p(ov[2]),
                            n_reservations=len(rn), res_node=_p(rn), res_cpu_milli=_p(rs[0]), res_mem_bytes=_p(rs[1]), res_gpu=_p(rs[2]))
        outs = [np.empty(max(n, 1), np.int64) for _ in range(3)]
        self._check(load().gp_build_reschedule_availability(self._h, C.byref(ui), *[_p(o) for o in outs]))
        return [o[:n] for o in outs]

    def prepare_cluster(self, alloc, overhead, res_node, res, zone_id=None, n_zones=1, name_rank=None, is_driver_candidate=None,
                        unschedulable=None, ready=None, driver_label_rank=None, executor_label_rank=None):
        """reservations -> availability -> priority orders -> snapshot, chained on the device.  -> (n_driver, n_executor)."""
        al = [_np(x, np.int64) for x in alloc]
        ov = [_np(x, np.int64) for x in overhead] if overhead is not None else [None] * 3
        rn = _np(res_node, np.int32)
        rs = [_np(x, np.int64) for x in res]
        n = len(al[0])
        ui = gp_usage_input(n_nodes=n, alloc_cpu_milli=_p(al[0]), alloc_mem_bytes=_p(al[1]), alloc_gpu=_p(al[2]),
                            overhead_cpu_milli=_p(ov[0]), overhead_mem_bytes=_p(ov[1]), overhead_gpu=_p(ov[2]),
                            n_reservations=len(rn), res_node=_p(rn), res_cpu_milli=_p(rs[0]), res_mem_bytes=_p(rs[1]), res_gpu=_p(rs[2]))
        arrs = [_np(zone_id, np.int32), _np(name_rank, np.int32), _np(is_driver_candidate, np.uint8), _np(unschedulable, np.uint8),
                _np(ready, np.uint8), _np(driver_label_rank, np.int32), _np(executor_label_rank, np.int32)]
        si = gp_sort_input(n_nodes=n, avail_cpu_milli=None, avail_mem_bytes=None, n_zones=n_zones, zone_id=_p(arrs[0]),
                           name_rank=_p(arrs[1]), is_driver_candidate=_p(arrs[2]), unschedulable=_p(arrs[3]), ready=_p(arrs[4]),
                           driver_label_rank=_p(arrs[5]), executor_label_rank=_p(arrs[6]))
        nd, ne = C.c_int32(0), C.c_int32(0)
        self._check(load().gp_prepare_cluster(self._h, C.byref(ui), C.byref(si), C.byref(nd), C.byref(ne)))
        self.n_nodes = n
        return nd.value, ne.value

    # ---- node priority order (NodeSorter.PotentialNodes) ---------------------------------------
    def potential_nodes(self, avail_cpu, avail_mem, zone_id=None, n_zones=1, name_rank=None, is_driver_candidate=None,
                        unschedulable=None, ready=None, driver_label_rank=None, executor_label_rank=None, avail_gpu=None):
        """-> (driver_order, executor_order) as int32 node-index arrays.  With avail_gpu given, self.undefined_ties is the
        number of adjacent pairs the reference's comparator leaves undefined (SURVEY App. B6)."""
        cpu, mem = _np(avail_cpu, np.int64), _np(avail_mem, np.int64)
        gpu = _np(avail_gpu, np.int64)
        n = len(cpu)
        arrs = [_np(zone_id, np.int32), _np(name_rank, np.int32), _np(is_driver_candidate, np.uint8), _np(unschedulable, np.uint8),
                _np(ready, np.uint8), _np(driver_label_rank, np.int32), _np(executor_label_rank, np.int32)]
        ties = C.c_int32(0)
        si = gp_sort_input(n_nodes=n, avail_cpu_milli=_p(cpu), avail_mem_bytes=_p(mem), n_zones=n_zones, zone_id=_p(arrs[0]),
                           name_rank=_p(arrs[1]), is_driver_candidate=_p(arrs[2]), unschedulable=_p(arrs[3]), ready=_p(arrs[4]),
                           driver_label_rank=_p(arrs[5]), executor_label_rank=_p(arrs[6]), avail_gpu=_p(gpu),
                           undefined_ties=C.addressof(ties))
        d = np.empty(max(n, 1), np.int32); e = np.empty(max(n, 1), np.int32)
        nd, ne = C.c_int32(0), C.c_int32(0)
        self._check(load().gp_potential_nodes(self._h, C.byref(si), _p(d), C.byref(nd), _p(e), C.byref(ne)))
        self.undefined_ties = ties.value
        return d[:nd.value].copy(), e[:ne.value].copy()

    # ---- packing -----------------------------------------------------------------------------
    def pack_batch(self, apps: dict, algo: int, mode: int = MODE_INDEPENDENT, out=None, wire=None):
        """apps: dict with drv_cpu, drv_mem, [drv_gpu], exe_cpu, exe_mem, [exe_gpu], count, [group], [young],
        [off].  Returns (driver_node[q], executor_nodes[sum count], off[q+1]).

        wire=None: the int64 layout through gp_pack_batch.  wire=dict(quantity_bits=32|64, mem_shift=.., node_bits=16|32,
        offsets=True|False) goes through gp_pack_batch_wire: with quantity_bits 32 the six quantity arrays of `apps` must
        ALREADY be int32 in wire units (millicores, bytes >> mem_shift, gpu units -- see compact_apps()); offsets=False
        passes exec_out_off = NULL (derived on the device)."""
        q = len(apps["count"])
        count = _np(apps["count"], np.int32)
        off = _np(apps.get("off"), np.int64)
        derive = wire is not None and not wire.get("offsets", True)
        if off is None and not (derive and out is not None):      # hot path (caller's buffers, device-derived offsets): no host cumsum
            off = np.zeros(q + 1, np.int64)
            np.cumsum(np.maximum(count, 0), out=off[1:])
        bits = 64 if wire is None else int(wire.get("quantity_bits", 64))
        qdt = np.int64 if bits == 64 else np.int32
        arrs = dict(
            drv_cpu=_np(apps["drv_cpu"], qdt), drv_mem=_np(apps["drv_mem"], qdt),
            drv_gpu=_np(apps.get("drv_gpu"), qdt),
            exe_cpu=_np(apps["exe_cpu"], qdt), exe_mem=_np(apps["exe_mem"], qdt),
            exe_gpu=_np(apps.get("exe_gpu"), qdt),
            group=_np(apps.get("group"), np.int32), young=_np(apps.get("young"), np.uint8))
        total = (int(off[-1]) if q else 0) if off is not None else len(out[1])
        node_bits = 32 if wire is None else int(wire.get("node_bits", 32))
        if out is None:
            driver_node = np.full(q, -9, np.int32)
            executor_nodes = np.full(max(total, 1), -9 if node_bits == 32 else 65535, np.int32 if node_bits == 32 else np.uint16)
        else:
            driver_node, executor_nodes = out
        if wire is None:
            a = gp_apps(n_apps=q, drv_cpu_milli=_p(arrs["drv_cpu"]), drv_mem_bytes=_p(arrs["drv_mem"]),
                        drv_gpu=_p(arrs["drv_gpu"]), exe_cpu_milli=_p(arrs["exe_cpu"]), exe_mem_bytes=_p(arrs["exe_mem"]),
                        exe_gpu=_p(arrs["exe_gpu"]), exe_count=_p(count), group=_p(arrs["group"]),
                        skip_if_no_fit=_p(arrs["young"]), exec_out_off=_p(off))
            r = gp_results(driver_node=_p(driver_node), executor_nodes=_p(executor_nodes),
                           executor_nodes_cap=len(executor_nodes))
            self._check(load().gp_pack_batch(self._h, C.byref(a), algo, mode, C.byref(r)))
        else:
            a = gp_apps_wire(n_apps=q, quantity_bits=bits, mem_shift=int(wire.get("mem_shift", 0)),
                             drv_cpu=_p(arrs["drv_cpu"]), drv_mem=_p(arrs["drv_mem"]), drv_gpu=_p(arrs["drv_gpu"]),
                             exe_cpu=_p(arrs["exe_cpu"]), exe_mem=_p(arrs["exe_mem"]), exe_gpu=_p(arrs["exe_gpu"]),
                             exe_count=_p(count), group=_p(arrs["group"]), skip_if_no_fit=_p(arrs["young"]),
                             exec_out_off=None if derive else _p(off))
            r = gp_results_wire(driver_node=_p(driver_node), executor_nodes=_p(executor_nodes),
                                executor_nodes_cap=len(executor_nodes), node_bits=node_bits)
            self._check(load().gp_pack_batch_wire(self._h, C.byref(a), algo, mode, C.byref(r)))
        return driver_node, executor_nodes[:total], off

    def set_schedulable(self, sched_cpu, sched_mem, sched_gpu=None):
        """NodeSchedulingMetadata.SchedulableResources of the current snapshot's nodes (needed by pack_batch_zones)."""
        c, m, g = _np(sched_cpu, np.int64), _np(sched_mem, np.int64), _np(sched_gpu, np.int64)
        self._check(load().gp_set_schedulable(self._h, _p(c), _p(m), _p(g)))

    def pack_batch_zones(self, apps: dict, algo: int):
        """single-az-tightly-pack / single-az-minimal-fragmentation for a batch: the snapshot's instance groups are the
        candidate zones.  -> (zone[q], driver_node[q], executor_nodes, off[q+1], avg_efficiency[q,4])."""
        q = len(apps["count"])
        count = _np(apps["count"], np.int32)
        off = np.zeros(q + 1, np.int64)
        np.cumsum(np.maximum(count, 0), out=off[1:])
        arrs = {k: _np(apps.get(k), np.int64) for k in ("drv_cpu", "drv_mem", "drv_gpu", "exe_cpu", "exe_mem", "exe_gpu")}
        total = int(off[-1]) if q else 0
        zone = np.full(q, -9, np.int32); drv = np.full(q, -9, np.int32)
        exe = np.full(max(total, 1), -9, np.int32); avg = np.zeros((max(q, 1), 4), np.float64)
        a = gp_apps(n_apps=q, drv_cpu_milli=_p(arrs["drv_cpu"]), drv_mem_bytes=_p(arrs["drv_mem"]), drv_gpu=_p(arrs["drv_gpu"]),
                    exe_cpu_milli=_p(arrs["exe_cpu"]), exe_mem_bytes=_p(arrs["exe_mem"]), exe_gpu=_p(arrs["exe_gpu"]),
                    exe_count=_p(count), group=None, skip_if_no_fit=None, exec_out_off=_p(off))
        r = gp_zone_results(zone=_p(zone), driver_node=_p(drv), executor_nodes=_p(exe), executor_nodes_cap=len(exe), avg_efficiency=_p(avg))
        self._check(load().gp_pack_batch_zones(self._h, C.byref(a), algo, C.byref(r)))
        return zone, drv, exe[:total], off, avg[:q]

    def pack_fifo_zones(self, apps: dict, algo: int, mode: int = 1):
        """fitEarlierDrivers with a single-AZ packer in one launch: `apps` is the queue in order (optional "young" = skip the
        driver instead of blocking the queue when it fits nowhere).  -> like pack_batch_zones; driver_node -2 = never evaluated."""
        q = len(apps["count"])
        count = _np(apps["count"], np.int32)
        off = np.zeros(q + 1, np.int64)
        np.cumsum(np.maximum(count, 0), out=off[1:])
        arrs = {k: _np(apps.get(k), np.int64) for k in ("drv_cpu", "drv_mem", "drv_gpu", "exe_cpu", "exe_mem", "exe_gpu")}
        young = _np(apps.get("young"), np.uint8)
        total = int(off[-1]) if q else 0
        zone = np.full(q, -9, np.int32); drv = np.full(q, -9, np.int32)
        exe = np.full(max(total, 1), -9, np.int32); avg = np.zeros((max(q, 1), 4), np.float64)
        a = gp_apps(n_apps=q, drv_cpu_milli=_p(arrs["drv_cpu"]), drv_mem_bytes=_p(arrs["drv_mem"]), drv_gpu=_p(arrs["drv_gpu"]),
                    exe_cpu_milli=_p(arrs["exe_cpu"]), exe_mem_bytes=_p(arrs["exe_mem"]), exe_gpu=_p(arrs["exe_gpu"]),
                    exe_count=_p(count), group=None, skip_if_no_fit=_p(young), exec_out_off=_p(off))
        r = gp_zone_results(zone=_p(zone), driver_node=_p(drv), executor_nodes=_p(exe), executor_nodes_cap=len(exe), avg_efficiency=_p(avg))
        self._check(load().gp_pack_fifo_zones(self._h, C.byref(a), algo, mode, C.byref(r)))
        return zone, drv, exe[:total], off, avg[:q]

    def reserve_placements(self, apps: dict, placed, subtract=True):
        """newResourceReservation for a packed batch -> dict of row arrays (app, slot, node, cpu, mem, gpu); with subtract the
        device-resident snapshot is charged with every reserved pod.  placed = (driver_node, executor_nodes, off)."""
        q = len(apps["count"])
        count = _np(apps["count"], np.int32)
        driver, execn, off = placed
        driver = _np(driver, np.int32); execn = _np(execn, np.int32); off = _np(off, np.int64)
        arrs = {k: _np(apps.get(k), np.int64) for k in ("drv_cpu", "drv_mem", "drv_gpu", "exe_cpu", "exe_mem", "exe_gpu")}
        rows = int(((driver >= 0) * (1 + np.maximum(count, 0).astype(np.int64))).sum()) if q else 0
        t = {k: np.zeros(max(rows, 1), np.int32) for k in ("app", "slot", "node")}
        t.update({k: np.zeros(max(rows, 1), np.int64) for k in ("cpu", "mem", "gpu")})
        a = gp_apps(n_apps=q, drv_cpu_milli=_p(arrs["drv_cpu"]), drv_mem_bytes=_p(arrs["drv_mem"]), drv_gpu=_p(arrs["drv_gpu"]),
                    exe_cpu_milli=_p(arrs["exe_cpu"]), exe_mem_bytes=_p(arrs["exe_mem"]), exe_gpu=_p(arrs["exe_gpu"]),
                    exe_count=_p(count), group=None, skip_if_no_fit=None, exec_out_off=_p(off))
        r = gp_results(driver_node=_p(driver), executor_nodes=_p(execn), executor_nodes_cap=len(execn))
        tab = gp_reservation_table(rows_cap=len(t["app"]), app=_p(t["app"]), slot=_p(t["slot"]), node=_p(t["node"]),
                                   cpu_milli=_p(t["cpu"]), mem_bytes=_p(t["mem"]), gpu=_p(t["gpu"]), n_rows=0)
        self._check(load().gp_reserve_placements(self._h, C.byref(a), C.byref(r), 1 if subtract else 0, C.byref(tab)))
        return {k: v[:tab.n_rows] for k, v in t.items()}

    def apply_usage_delta(self, node, cpu, mem, gpu=None, sign=1):
        n, c, m, g = _np(node, np.int32), _np(cpu, np.int64), _np(mem, np.int64), _np(gpu, np.int64)
        self._check(load().gp_apply_usage_delta(self._h, len(n), _p(n), _p(c), _p(m), _p(g), sign))

    # ---- bound calls: what a shim does -- marshal the argument structs ONCE over its long-lived buffers, then one FFI call
    # per Predicate (the numpy / ctypes marshalling of set_snapshot() / pack_batch() costs more than a small batch's kernels)
    def bind_snapshot(self, avail_cpu, avail_mem, avail_gpu, exec_order, drv_order, exec_off, drv_off):
        """-> zero-argument callable running gp_set_snapshot on these (caller-owned, stable) arrays."""
        keep = [_np(avail_cpu, np.int64), _np(avail_mem, np.int64), _np(avail_gpu, np.int64), _np(exec_order, np.int32),
                _np(drv_order, np.int32), _np(exec_off, np.int32), _np(drv_off, np.int32)]
        n = gp_nodes(n_nodes=len(keep[0]), avail_cpu_milli=_p(keep[0]), avail_mem_bytes=_p(keep[1]), avail_gpu=_p(keep[2]),
                     n_groups=len(keep[5]) - 1, exec_off=_p(keep[5]), exec_order=_p(keep[3]), drv_off=_p(keep[6]), drv_order=_p(keep[4]))
        fn, h, ref = load().gp_set_snapshot, self._h, C.byref(n)
        self.n_nodes = len(keep[0])

        def call(_keep=(keep, n)):
            st = fn(h, ref)
            if st != 0:
                self._check(st)
        return call

    def bind_batch(self, apps: dict, algo: int, mode: int, out, wire: dict):
        """-> zero-argument callable running gp_pack_batch_wire on these (caller-owned, stable) arrays; results land in `out`."""
        bits = int(wire.get("quantity_bits", 64))
        qdt = np.int64 if bits == 64 else np.int32
        q = len(apps["count"])
        keep = {k: _np(apps.get(k), qdt) for k in ("drv_cpu", "drv_mem", "drv_gpu", "exe_cpu", "exe_mem", "exe_gpu")}
        keep["count"] = _np(apps["count"], np.int32)
        keep["group"] = _np(apps.get("group"), np.int32)
        keep["young"] = _np(apps.get("young"), np.uint8)
        keep["off"] = _np(apps.get("off"), np.int64) if wire.get("offsets", True) else None
        if wire.get("offsets", True) and keep["off"] is None:
            raise ValueError("bind_batch: wire.offsets is set but apps has no 'off'")
        driver_node, executor_nodes = out
        a = gp_apps_wire(n_apps=q, quantity_bits=bits, mem_shift=int(wire.get("mem_shift", 0)),
                         drv_cpu=_p(keep["drv_cpu"]), drv_mem=_p(keep["drv_mem"]), drv_gpu=_p(keep["drv_gpu"]),
                         exe_cpu=_p(keep["exe_cpu"]), exe_mem=_p(keep["exe_mem"]), exe_gpu=_p(keep["exe_gpu"]),
                         exe_count=_p(keep["count"]), group=_p(keep["group"]), skip_if_no_fit=_p(keep["young"]),
                         exec_out_off=_p(keep["off"]))
        r = gp_results_wire(driver_node=_p(driver_node), executor_nodes=_p(executor_nodes),
                            executor_nodes_cap=len(executor_nodes), node_bits=int(wire.get("node_bits", 32)))
        fn, h, ra, rr = load().gp_pack_batch_wire, self._h, C.byref(a), C.byref(r)

        def call(_keep=(keep, a, r, out)):
            st = fn(h, ra, algo, mode, rr)
            if st != 0:
                self._check(st)
        return call

    def pack_one(self, algo, drv, exe, count):
        """binpack.SparkBinPackFunction for one app -> (has_capacity, driver_node, executor_nodes)."""
        has = C.c_int32(0); d = C.c_int32(-1)
        en = np.full(max(count, 1), -9, np.int32)
        self._check(load().gp_pack_one(self._h, algo, int(drv[0]), int(drv[1]), int(drv[2]), int(exe[0]), int(exe[1]),
                                       int(exe[2]), int(count), C.byref(has), C.byref(d), _p(en)))
        return bool(has.value), d.value, en[:count] if has.value else en[:0]

    def stats(self) -> dict:
        s = gp_stats()
        self._check(load().gp_last_stats(self._h, C.byref(s)))
        return {"nodes_scanned": s.nodes_scanned, "drivers_tried": s.drivers_tried, "kernel_launches": s.kernel_launches,
                "pack_kernel_ns": s.pack_kernel_ns, "prep_kernel_ns": s.prep_kernel_ns,
                "scan_path_apps": s.scan_path_apps, "scan_path_nodes": s.scan_path_nodes}

    # ---- device-resident (torch tensors on this context's device) ----------------------------
    def stream_handle(self) -> int:
        return load().gp_stream(self._h) or 0

    def synchronize(self):
        self._check(load().gp_synchronize(self._h))

    def set_snapshot_device(self, cpu, mem, gpu, exec_off, exec_order, drv_off, drv_order, stream: int = 0):
        """All arguments are torch CUDA tensors (int64 / int32); kept alive by the caller."""
        n = gp_nodes(n_nodes=cpu.numel(), avail_cpu_milli=cpu.data_ptr(), avail_mem_bytes=mem.data_ptr(),
                     avail_gpu=gpu.data_ptr() if gpu is not None else None, n_groups=exec_off.numel() - 1,
                     exec_off=exec_off.data_ptr(), exec_order=exec_order.data_ptr(), drv_off=drv_off.data_ptr(),
                     drv_order=drv_order.data_ptr())
        self._check(load().gp_set_snapshot_device(self._h, C.byref(n), exec_order.numel(), drv_order.numel(),
                                                  stream or None))
        self.n_nodes = cpu.numel()

    def pack_batch_device(self, t: dict, algo: int, mode: int, driver_node, executor_nodes, stream: int = 0):
        """t: dict of torch CUDA tensors (drv_cpu, drv_mem, [drv_gpu], exe_cpu, exe_mem, [exe_gpu], count, [group],
        [young], off).  Asynchronous on `stream` (0 = the context's stream)."""
        def dp(name):
            v = t.get(name)
            return v.data_ptr() if v is not None else None
        a = gp_apps(n_apps=t["count"].numel(), drv_cpu_milli=dp("drv_cpu"), drv_mem_bytes=dp("drv_mem"),
                    drv_gpu=dp("drv_gpu"), exe_cpu_milli=dp("exe_cpu"), exe_mem_bytes=dp("exe_mem"),
                    exe_gpu=dp("exe_gpu"), exe_count=dp("count"), group=dp("group"), skip_if_no_fit=dp("young"),
                    exec_out_off=dp("off"))
        r = gp_results(driver_node=driver_node.data_ptr(), executor_nodes=executor_nodes.data_ptr(),
                       executor_nodes_cap=executor_nodes.numel())
        self._check(load().gp_pack_batch_device(self._h, C.byref(a), algo, mode, C.byref(r), stream or None))


class MultiGangPacker:
    """gp_multi: one host process, several GPUs (or several contexts on one GPU).  Same call shapes as GangPacker."""

    def __init__(self, devices):
        L = load()
        self._h = C.c_void_p()
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        st = L.gp_multi_create(C.byref(self._h), dev.ctypes.data, len(dev))
        if st != 0:
            raise GangpackError(st, (L.gp_last_error(None) or b"").decode())
        self.n_devices = len(dev)
        self._pinned = []

    def close(self):
        if getattr(self, "_h", None):
            for ctx, ptr in self._pinned:
                load().gp_free_pinned(ctx, ptr)
            self._pinned = []
            load().gp_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st):
        if st != 0:
            raise GangpackError(st, (load().gp_multi_last_error(self._h) or b"").decode())

    def pinned(self, shape, dtype) -> np.ndarray:
        """Pinned host memory (portable: usable by every device of the handle)."""
        dt = np.dtype(dtype)
        n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
        nbytes = max(n * dt.itemsize, 1)
        ptr = C.c_void_p()
        ctx = load().gp_multi_ctx(self._h, 0)
        st = load().gp_alloc_pinned(ctx, nbytes, C.byref(ptr))
        if st != 0:
            raise GangpackError(st, (load().gp_last_error(ctx) or b"").decode())
        self._pinned.append((ctx, ptr))
        buf = (C.c_char * nbytes).from_address(ptr.value)
        return np.frombuffer(buf, dtype=dt, count=n).reshape(shape)

    def set_snapshot(self, avail_cpu, avail_mem, avail_gpu, exec_order, drv_order, exec_off=None, drv_off=None):
        cpu, mem, gpu = _np(avail_cpu, np.int64), _np(avail_mem, np.int64), _np(avail_gpu, np.int64)
        eo, do = _np(exec_order, np.int32), _np(drv_order, np.int32)
        eoff = _np(exec_off if exec_off is not None else [0, len(eo)], np.int32)
        doff = _np(drv_off if drv_off is not None else [0, len(do)], np.int32)
        n = gp_nodes(n_nodes=len(cpu), avail_cpu_milli=_p(cpu), avail_mem_bytes=_p(mem), avail_gpu=_p(gpu),
                     n_groups=len(eoff) - 1, exec_off=_p(eoff), exec_order=_p(eo), drv_off=_p(doff), drv_order=_p(do))
        self._check(load().gp_multi_set_snapshot(self._h, C.byref(n)))
        self.n_nodes, self.n_groups = len(cpu), len(eoff) - 1

    def get_snapshot(self):
        cpu = np.empty(self.n_nodes, np.int64); mem = np.empty(self.n_nodes, np.int64); gpu = np.empty(self.n_nodes, np.int64)
        self._check(load().gp_multi_get_snapshot(self._h, _p(cpu), _p(mem), _p(gpu)))
        return cpu, mem, gpu

    def group_owner(self):
        o = np.empty(self.n_groups, np.int32)
        self._check(load().gp_multi_group_owner(self._h, _p(o)))
        return o

    def pack_batch(self, apps: dict, algo: int, mode: int = MODE_INDEPENDENT, out=None, wire=None):
        """Same contract as GangPacker.pack_batch (wire=None -> int64 quantities, offsets given, int32 node indices)."""
        wire = dict(wire or dict(quantity_bits=64, node_bits=32, offsets=True))
        q = len(apps["count"])
        count = _np(apps["count"], np.int32)
        off = _np(apps.get("off"), np.int64)
        derive = not wire.get("offsets", True)
        if off is None and not (derive and out is not None):      # hot path (caller's buffers, device-derived offsets): no host cumsum
            off = np.zeros(q + 1, np.int64)
            np.cumsum(np.maximum(count, 0), out=off[1:])
        bits = int(wire.get("quantity_bits", 64))
        qdt = np.int64 if bits == 64 else np.int32
        arrs = {k: _np(apps.get(k), qdt) for k in ("drv_cpu", "drv_mem", "drv_gpu", "exe_cpu", "exe_mem", "exe_gpu")}
        grp, young = _np(apps.get("group"), np.int32), _np(apps.get("young"), np.uint8)
        total = (int(off[-1]) if q else 0) if off is not None else len(out[1])
        node_bits = int(wire.get("node_bits", 32))
        if out is None:
            driver_node = np.full(q, -9, np.int32)
            executor_nodes = np.full(max(total, 1), -9 if node_bits == 32 else 65535, np.int32 if node_bits == 32 else np.uint16)
        else:
            driver_node, executor_nodes = out
        a = gp_apps_wire(n_apps=q, quantity_bits=bits, mem_shift=int(wire.get("mem_shift", 0)),
                         drv_cpu=_p(arrs["drv_cpu"]), drv_mem=_p(arrs["drv_mem"]), drv_gpu=_p(arrs["drv_gpu"]),
                         exe_cpu=_p(arrs["exe_cpu"]), exe_mem=_p(arrs["exe_mem"]), exe_gpu=_p(arrs["exe_gpu"]),
                         exe_count=_p(count), group=_p(grp), skip_if_no_fit=_p(young),
                         exec_out_off=None if derive else _p(off))
        r = gp_results_wire(driver_node=_p(driver_node), executor_nodes=_p(executor_nodes),
                            executor_nodes_cap=len(executor_nodes), node_bits=node_bits)
        self._check(load().gp_multi_pack_batch(self._h, C.byref(a), algo, mode, C.byref(r)))
        return driver_node, executor_nodes[:total], off
