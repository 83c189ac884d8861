"""ctypes binding of libb200serve.so (include/b200serve.h).

There is no CPU fallback: if the library is missing, or no GPU is present when a device call is made,
a `NativeError` is raised.  Loading the library itself does not need a GPU (the CPU test-suite checks
that every symbol of the header is exported).
"""

import ctypes as C
import collections
import os
import threading
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200serve.so")

# mirrors of the header's constants
OUT_COPY, OUT_ONEHOT = 0, 1
LINK_IDENTITY, LINK_BINARY_GT, LINK_BINARY_GE, LINK_ARGMAX = 0, 1, 2, 3
VOTE_NONE, VOTE_MEAN, VOTE_MAJORITY = 0, 1, 2
ROW_NONFINITE_INPUT, ROW_BAD_LABEL, ROW_UNKNOWN_KEY = 1, 2, 4
CMP_LE, CMP_LT = 0, 1          # left when x <= threshold (scikit-learn, LightGBM) | x < threshold (xgboost)
NAN_ERROR, NAN_DEFAULT_CHILD = 0, 1
COL_F32, COL_I32, COL_I64 = 0, 1, 2
STAT_F32, STAT_I32, STAT_I32_NAT, STAT_BOOL, STAT_DT, STAT_ROW = 0, 1, 2, 3, 4, 5
STAT_RANKS, STAT_BINS = 6, 20
DATE_PARTS = {"year": 0, "month": 1, "day": 2, "hour": 3, "minute": 4, "second": 5, "day_of_week": 6, "dayofweek": 6,
              "weekday": 6, "day_of_year": 7, "dayofyear": 7, "quarter": 8, "is_leap_year": 9, "days_in_month": 10,
              "daysinmonth": 10, "is_month_start": 11, "is_month_end": 12, "is_quarter_start": 13, "is_quarter_end": 14,
              "is_year_start": 15, "is_year_end": 16, "week": 17, "weekofyear": 17}
DATE_BOOL_PARTS = {9, 11, 12, 13, 14, 15, 16}


class NativeError(RuntimeError):
    """the CUDA engine is unavailable or a C-ABI call failed"""


class Stats(C.Structure):
    _fields_ = [("rows", C.c_int64), ("h2d_ms", C.c_float), ("kernel_ms", C.c_float), ("d2h_ms", C.c_float),
                ("queue_us", C.c_float), ("kernels", C.c_int32), ("nonfinite_rows", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ColSum(C.Structure):
    """b2s_colsum: pass 0 of the feature-set statistics, one per described column"""
    _fields_ = [("count", C.c_int64), ("missing", C.c_int64), ("ones", C.c_int64), ("pos_inf", C.c_int32),
                ("neg_inf", C.c_int32), ("sum", C.c_double), ("min_bits", C.c_int64), ("max_bits", C.c_int64),
                ("first_bits", C.c_int64), ("first_missing", C.c_int32), ("pad_", C.c_int32)]


class DevInfo(C.Structure):
    _fields_ = [("ordinal", C.c_int32), ("sm_count", C.c_int32), ("cc_major", C.c_int32), ("cc_minor", C.c_int32),
                ("total_mem", C.c_int64), ("l2_bytes", C.c_int64), ("smem_per_block_optin", C.c_int64),
                ("name", C.c_char * 128)]


_vp, _i32, _i64, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
_pi32, _pf32, _pf64 = C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_double)

# name -> (restype, argtypes); the single source of truth for the exported surface
SIGNATURES = {
    "b2s_version": (C.c_int, []),
    "b2s_last_error": (C.c_char_p, []),
    "b2s_init": (C.c_int, [C.c_int, C.c_char_p]),
    "b2s_shutdown": (C.c_int, []),
    "b2s_device_info": (C.c_int, [C.POINTER(DevInfo)]),
    "b2s_launch_count": (_i64, []),
    "b2s_plan_create": (C.c_int, [_i32, C.POINTER(_vp)]),
    "b2s_plan_destroy": (C.c_int, [_vp]),
    "b2s_plan_set_impute": (C.c_int, [_vp, _pi32, _pf32, _i32]),
    "b2s_plan_add_value_map": (C.c_int, [_vp, _i32, _pf32, _pf32, _i32]),
    "b2s_plan_add_range_map": (C.c_int, [_vp, _i32, _pf32, _pf32, _pf32, _i32]),
    "b2s_plan_set_output_schema": (C.c_int, [_vp, _pi32, _pi32, _pf32, _i32]),
    "b2s_plan_add_linear_model": (C.c_int, [_vp, _pf64, _pf64, _i32, _i32, _pi32, _i32]),
    "b2s_plan_add_tree_model": (C.c_int, [_vp, _i32, _pi32, _pi32, _pf32, _pi32, _pi32, _pf64, _pi32, _pf64, _pf64,
                                          _i32, _i32, _pi32, _i32]),
    "b2s_plan_add_tree_model_ex": (C.c_int, [_vp, _i32, _pi32, _pi32, _pf32, _pi32, _pi32, _pf64, _pi32, _pf64, _pf64,
                                             _i32, _i32, _pi32, _i32, _i32, C.POINTER(C.c_uint8), _i32]),
    "b2s_plan_set_vote": (C.c_int, [_vp, _i32, _pf64, _i32]),
    "b2s_plan_finalize": (C.c_int, [_vp]),
    "b2s_plan_out_info": (C.c_int, [_vp, _pi32, _pi32]),
    "b2s_plan_kernel": (C.c_char_p, [_vp]),
    "b2s_run_device": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "b2s_run_host": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _vp, C.POINTER(Stats)]),
    "b2s_submit": (C.c_int, [_vp, _vp, _i64, _i64, C.POINTER(_u64)]),
    "b2s_wait": (C.c_int, [_vp, _u64, _vp, _i64, _vp, C.POINTER(Stats)]),
    "b2s_flush": (C.c_int, [_vp]),
    "b2s_plan_set_ring": (C.c_int, [_vp, _i32, _i64, _i32]),
    "b2s_ring_bench": (C.c_int, [_vp, _vp, _i64, _i64, _i32, _i32, C.c_double, C.POINTER(_i64), C.POINTER(C.c_double),
                                 C.POINTER(C.c_double)]),
    "b2s_plan_set_merge_targets": (C.c_int, [_vp, C.POINTER(_vp), _i32, _i64]),
    "b2s_comm_create": (C.c_int, [_i32, _i32, _i64, _i32, C.POINTER(_vp)]),
    "b2s_comm_handle": (C.c_int, [_vp, _vp]),
    "b2s_comm_connect": (C.c_int, [_vp, _vp]),
    "b2s_plan_attach_comm": (C.c_int, [_vp, _vp]),
    "b2s_comm_wait": (C.c_int, [_vp, _vp, C.POINTER(_vp), C.POINTER(C.c_uint32)]),
    "b2s_comm_wait_lag": (C.c_int, [_vp, _vp, C.c_int32, C.POINTER(_vp), C.POINTER(C.c_uint32)]),
    "b2s_comm_set_fused_wait": (C.c_int, [_vp, C.c_int32]),
    "b2s_comm_check": (C.c_int, [_vp]),
    "b2s_comm_destroy": (C.c_int, [_vp]),
    "b2s_ipc_export": (C.c_int, [_vp, _vp]),
    "b2s_ipc_open": (C.c_int, [_vp, C.POINTER(_vp)]),
    "b2s_ipc_close": (C.c_int, [_vp]),
    "b2s_alloc_pinned": (_vp, [C.c_size_t]),
    "b2s_free_pinned": (C.c_int, [_vp]),
    "b2s_device_alloc": (_vp, [C.c_size_t]),
    "b2s_device_free": (C.c_int, [_vp]),
    "b2s_memcpy_h2d": (C.c_int, [_vp, _vp, C.c_size_t]),
    "b2s_memcpy_d2h": (C.c_int, [_vp, _vp, C.c_size_t]),
    "b2s_device_sync": (C.c_int, []),
    "b2s_time_device": (C.c_int, [_vp, C.POINTER(_vp), _i32, _i64, _i64, _vp, _i32, _pf32]),
    # columnar ingest
    "b2s_cols_create": (C.c_int, [_i32, C.POINTER(_vp)]),
    "b2s_cols_destroy": (C.c_int, [_vp]),
    "b2s_cols_add_copy": (C.c_int, [_vp, _i32, _i32, _i32, C.c_float, _i32, _i32, C.c_double, C.c_double, _pi32, _pi32]),
    "b2s_cols_add_range_map": (C.c_int, [_vp, _i32, _i32, _i32, C.c_float, _pf64, _pf64, _pf64, _i32, _i32, C.c_double,
                                         C.c_double, _pi32, _pi32, _pi32]),
    "b2s_cols_add_value_map": (C.c_int, [_vp, _i32, _i32, _i32, C.c_float, _pf64, _pf64, _i32, _i32, C.c_double, C.c_double,
                                         _pi32, _pi32, _pi32]),
    "b2s_cols_add_onehot": (C.c_int, [_vp, _i32, _i32, _i32, C.c_float, _pf64, _i32, _pi32, _pi32]),
    "b2s_cols_add_date_part": (C.c_int, [_vp, _i32, _i32, _pi32, _pi32]),
    "b2s_cols_finalize": (C.c_int, [_vp]),
    "b2s_cols_info": (C.c_int, [_vp, _pi32, _pi32]),
    "b2s_cols_run_device": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _vp, _vp]),
    "b2s_cols_run_host": (C.c_int, [_vp, C.POINTER(_vp), _i64, C.POINTER(_vp), C.POINTER(_u64), C.POINTER(Stats)]),
    "b2s_cols_stats_begin": (C.c_int, [_vp, _vp, _i64, _i64, _pi32, _pi32, _i32, _vp, C.POINTER(Stats)]),
    "b2s_cols_stats_finish": (C.c_int, [_vp, _pf64, _pi32, _pf64, C.POINTER(_i64), _pf64, C.POINTER(_i64), C.POINTER(_i64),
                                        C.POINTER(Stats)]),
    "b2s_cols_stats_timing": (C.c_int, [_vp, _pf32, C.POINTER(_i64), _pi32, _pi32]),
    # online feature table
    "b2s_table_create": (C.c_int, [C.POINTER(_i64), _i64, _pf32, _i32, _pf32, C.POINTER(_vp)]),
    "b2s_table_destroy": (C.c_int, [_vp]),
    "b2s_table_info": (C.c_int, [_vp, C.POINTER(_i64), _pi32, C.POINTER(_i64)]),
    "b2s_table_lookup_device": (C.c_int, [_vp, _vp, _i64, _vp, _i64, _vp, _vp]),
    "b2s_table_lookup_host": (C.c_int, [_vp, C.POINTER(_i64), _i64, _pf32, _pi32, C.POINTER(Stats)]),
    "b2s_table_enrich_device": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "b2s_table_enrich_host": (C.c_int, [_vp, _vp, C.POINTER(_i64), _i64, _vp, _i64, _pi32, C.POINTER(Stats)]),
    "b2s_table_time_device": (C.c_int, [_vp, C.POINTER(_vp), _i32, _i64, _vp, _i64, _vp, _i32, _pf32]),
    "b2s_hash_strings": (C.c_int, [C.c_char_p, C.POINTER(_i64), _i64, C.POINTER(_i64)]),
    # body codec
    "b2s_json_parse_inputs": (C.c_int, [C.c_char_p, _i64, _pf32, _i64, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64),
                                        C.POINTER(_i64)]),
    "b2s_json_format_outputs": (C.c_int, [_vp, _i32, _i64, _i64, _i32, C.c_char_p, _i64, C.POINTER(_i64)]),
    "b2s_cols_time_device": (C.c_int, [_vp, C.POINTER(_vp), _i32, _i64, _i64, _vp, _i64, _vp, _i32, _pf32]),
}

_lib = None
_lock = threading.Lock()
_inited = False


def load():
    """dlopen the library (no GPU needed) and declare every signature"""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeError(
                    f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(nvcc, sm_100a). mlrun_b200 has no CPU fallback for device steps."
                )
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        msg = load().b2s_last_error()
        raise NativeError(f"b200serve error {rc}: {msg.decode() if msg else ''}")


def init(device=None, cfg=None):
    """bring up the device once per process (device ordinal defaults to LOCAL_RANK or 0)"""
    global _inited
    lib = load()
    if _inited:
        return lib
    with _lock:
        if not _inited:
            if device is None:
                device = int(os.environ.get("LOCAL_RANK", "0"))
            cfg = cfg or os.environ.get("B200SERVE_CFG", "")
            check(lib.b2s_init(int(device), cfg.encode() if cfg else None))
            _inited = True
    return lib


def device_info():
    lib = init()
    info = DevInfo()
    check(lib.b2s_device_info(C.byref(info)))
    return {"name": info.name.decode(), "sm_count": info.sm_count, "cc": (info.cc_major, info.cc_minor),
            "total_mem": info.total_mem, "l2_bytes": info.l2_bytes, "smem_optin": info.smem_per_block_optin}


def launch_count():
    return int(load().b2s_launch_count())


def ptr(arr):
    """address of a numpy array's first element, 3x cheaper than `arr.ctypes.data` (which builds a helper object per call:
    1.2 us, three of them per serving call); read-only, empty and non-contiguous arrays take the ordinary route"""
    try:
        return C.addressof(C.c_char.from_buffer(arr))
    except (TypeError, ValueError):
        return arr.ctypes.data


def _p(arr, ctype):
    return arr.ctypes.data_as(C.POINTER(ctype)) if arr is not None else None


class DeviceBuffer:
    """a cudaMalloc'd buffer owned by the library (ctypes callers need no other CUDA binding)"""

    def __init__(self, nbytes):
        lib = init()
        self.nbytes = int(nbytes)
        self.ptr = lib.b2s_device_alloc(self.nbytes)
        if not self.ptr:
            raise NativeError(f"device alloc of {nbytes} bytes failed: {lib.b2s_last_error().decode()}")

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        check(load().b2s_memcpy_h2d(self.ptr, arr.ctypes.data, arr.nbytes))
        return self

    def download(self, dtype, shape):
        out = np.empty(shape, dtype=dtype)
        check(load().b2s_memcpy_d2h(out.ctypes.data, self.ptr, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            load().b2s_device_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def ipc_export(dptr):
    """64-byte CUDA IPC handle of a buffer from DeviceBuffer / b2s_device_alloc"""
    buf = C.create_string_buffer(64)
    check(load().b2s_ipc_export(dptr, buf))
    return bytes(buf.raw)


def ipc_open(handle):
    out = C.c_void_p()
    check(load().b2s_ipc_open(C.create_string_buffer(handle, 64), C.byref(out)))
    return out.value


def pinned_empty(shape, dtype=np.float32):
    """numpy array over cudaMallocHost memory (kept alive by the returned array's base object)"""
    lib = init()
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = lib.b2s_alloc_pinned(max(nbytes, 1))
    if not ptr:
        raise NativeError("pinned alloc failed")
    buf = (C.c_char * max(nbytes, 1)).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    # the block goes back to the driver when the last array over it is collected (arrays keep `buf` alive as their base)
    weakref.finalize(buf, _free_pinned, ptr)
    return arr


def _free_pinned(ptr):
    try:
        if _lib is not None:
            _lib.b2s_free_pinned(ptr)
    except Exception:
        pass


class _Lease:
    """keeps a pinned block out of the pool while any numpy array over it is alive (the arrays' base buffer holds it)"""

    def __init__(self, pool, ptr, size):
        self.pool, self.ptr, self.size = pool, ptr, size

    def __del__(self):
        # may run inside a garbage-collection pass triggered while take() holds the pool lock on this very thread:
        # only append to a deque here (atomic, lock free); take() drains it
        try:
            self.pool._returned.append((self.ptr, self.size))
        except Exception:
            pass


class PinnedPool:
    """cudaMallocHost blocks for results that go straight into numpy / DataFrame columns: D2H copies into pinned memory run
    at PCIe speed, and the block is reused once the arrays built over it are garbage collected.  At most `max_blocks`
    blocks exist; beyond that `take` returns None and the caller uses pageable memory."""

    def __init__(self, max_blocks=6, granule=1 << 20):
        self.max_blocks, self.granule = max_blocks, granule
        self._free = {}
        self._n = 0
        self._mu = threading.RLock()
        self._returned = collections.deque()  # blocks whose arrays died (filled by _Lease.__del__ without the lock)

    def take(self, nbytes):
        size = max(self.granule, (int(nbytes) + self.granule - 1) // self.granule * self.granule)
        with self._mu:
            self._drain()
            ptrs = self._free.get(size)
            ptr = ptrs.pop() if ptrs else None
            if ptr is None:
                if self._n >= self.max_blocks:
                    victim = next((s for s, p in self._free.items() if p), None)  # a free block of another size makes room
                    if victim is None:
                        return None
                    load().b2s_free_pinned(self._free[victim].pop())
                    self._n -= 1
                ptr = init().b2s_alloc_pinned(size)
                if not ptr:
                    return None
                self._n += 1
        buf = (C.c_char * size).from_address(ptr)
        buf._lease = _Lease(self, ptr, size)
        return buf

    def _drain(self):
        while True:
            try:
                ptr, size = self._returned.popleft()
            except IndexError:
                return
            self._free.setdefault(size, []).append(ptr)

    def _give_back(self, ptr, size):
        self._returned.append((ptr, size))


PINNED = PinnedPool()
