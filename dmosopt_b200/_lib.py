"""ctypes binding of libdmosopt_b200.so (include/dmosopt_b200.h).

Thin layer: argument marshalling and error translation only.  Every function
takes/returns NumPy arrays (host) -- or, for inputs, anything exposing a CUDA
device pointer through ``data_ptr()`` (torch tensors) when the caller keeps
data resident.  There is deliberately NO CPU fallback: if the CUDA library is
missing or no GPU is present the import of the library / creation of the
context raises.
"""

import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdmosopt_b200.so")

METRIC_NONE, METRIC_CROWDING, METRIC_EUCLIDEAN = 0, 1, 2
KERNEL_MATERN52, KERNEL_RBF = 0, 1
GP_FP64, GP_TENSOR, GP_AUTO = 0, 1, 2
HV_MAX_OBJECTIVES = 8  # dmo_hypervolume: exact, chain sums for M <= 5 (csrc/hv.cu), limit-set recursion for 6 .. 8 (csrc/hv_many.cu)

_c_i64 = ctypes.c_int64
_c_u64 = ctypes.c_uint64
_c_int = ctypes.c_int
_c_dbl = ctypes.c_double
_vp = ctypes.c_void_p

# exported symbols -> (restype, argtypes); checked against the header by tests/test_abi.py
_SIGNATURES = {
    "dmo_version": (_c_int, []),
    "dmo_create": (_c_int, [_c_int, ctypes.POINTER(_vp)]),
    "dmo_destroy": (_c_int, [_vp]),
    "dmo_last_error": (ctypes.c_char_p, [_vp]),
    "dmo_synchronize": (_c_int, [_vp]),
    "dmo_stream": (_vp, [_vp]),
    "dmo_launch_count": (_c_i64, [_vp]),
    "dmo_sm_count": (_c_int, [_vp]),
    "dmo_timer_begin": (_c_int, [_vp]),
    "dmo_timer_end": (_c_int, [_vp, ctypes.POINTER(ctypes.c_float)]),
    "dmo_host_alloc": (_c_int, [ctypes.POINTER(_vp), _c_u64]),
    "dmo_host_free": (_c_int, [_vp]),
    "dmo_device_alloc": (_c_int, [_vp, ctypes.POINTER(_vp), _c_u64]),
    "dmo_device_free": (_c_int, [_vp, _vp]),
    "dmo_memcpy": (_c_int, [_vp, _vp, _vp, _c_u64]),
    "dmo_flush_l2": (_c_int, [_vp]),
    "dmo_transfer_bytes": (_c_int, [_vp, ctypes.POINTER(_c_u64), ctypes.POINTER(_c_u64)]),
    "dmo_profile_enable": (_c_int, [_vp, _c_int]),
    "dmo_profile_report": (_c_int, [_vp, ctypes.c_char_p, _c_u64]),
    "dmo_round_f32": (_c_int, [_vp, _vp, _c_i64]),
    "dmo_rank_nd": (_c_int, [_vp, _vp, _c_i64, _c_int, _vp]),
    "dmo_crowding_distance": (_c_int, [_vp, _vp, _c_i64, _c_int, _vp]),
    "dmo_euclidean_distance": (_c_int, [_vp, _vp, _c_i64, _c_int, _vp]),
    "dmo_order_mo": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _vp, _c_int, _vp, _vp, _vp]),
    "dmo_remove_worst": (_c_int, [_vp, _vp, _vp, _c_i64, _c_int, _c_int, _c_int, _vp, _c_int, _c_i64, _vp, _vp, _vp, _vp]),
    "dmo_remove_worst_pair": (_c_int, [_vp, _vp, _vp, _c_i64, _vp, _vp, _c_i64, _c_int, _c_int, _c_int, _c_i64, _vp, _vp, _vp, _vp]),
    "dmo_tournament": (_c_int, [_vp, _vp, _vp, _c_i64, _c_i64, _c_u64, _c_u64, _vp, _vp]),
    "dmo_mutation_u": (_c_int, [_vp, _vp, _vp, _c_i64, _c_int, _vp, _vp, _vp, _c_dbl, _vp]),
    "dmo_sbx_u": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_int, _vp, _vp, _vp, _vp, _vp]),
    "dmo_nsga2_plan_length": (_c_i64, [_c_i64, _c_dbl, _c_dbl]),
    "dmo_nsga2_generate": (
        _c_int,
        [_vp, _vp, _c_i64, _c_int, _vp, _c_i64, _c_i64, _c_dbl, _c_dbl, _c_dbl, _vp, _vp, _vp, _vp, _c_u64, _c_u64, _vp, _vp, _vp, _vp],
    ),
    "dmo_gp_create": (_c_int, [_vp, _c_i64, _c_int, _c_int, _c_int, _vp, _vp, _vp, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "dmo_gp_destroy": (_c_int, [_vp, _vp]),
    "dmo_gp_fit": (_c_int, [_vp, _c_i64, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp, _c_dbl, _vp, _vp, _vp]),
    "dmo_gp_set_linear_mean": (_c_int, [_vp, _vp, _vp, _vp]),
    "dmo_gp_predict": (_c_int, [_vp, _vp, _vp, _c_i64, _vp, _vp, _c_int]),
    "dmo_gp_auto_info": (_c_int, [_vp, _vp, ctypes.POINTER(_c_int), ctypes.POINTER(_c_int), ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl),
                                  ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_i64)]),
    "dmo_nsga2_step": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _vp, _vp, _vp, _vp, _c_u64, _c_u64,
                                _c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp]),
    "dmo_hypervolume": (_c_int, [_vp, _vp, _c_i64, _c_int, _vp, ctypes.POINTER(_c_dbl)]),
    "dmo_hypervolume_ranked": (_c_int, [_vp, _vp, _c_i64, _c_int, _vp, _vp, ctypes.POINTER(_c_dbl)]),
    "dmo_ehvi_select": (_c_int, [_vp, _vp, _c_i64, _vp, _vp, _c_i64, _c_int, _vp, _c_int, _c_i64, _vp, _vp]),
    "dmo_get_duplicates": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_dbl, _vp]),
    "dmo_get_duplicates_pair": (_c_int, [_vp, _vp, _c_i64, _vp, _c_i64, _c_int, _c_dbl, _vp]),
    "dmo_age_survival": (_c_int, [_vp, _vp, _vp, _c_i64, _c_int, _c_dbl, _vp, _c_int, _vp]),
    "dmo_smpso_velocity": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_int, _c_i64, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_dbl, _c_dbl, _c_dbl, _vp, _vp, _vp]),
    "dmo_mutate_groups": (_c_int, [_vp, _vp, _c_i64, _c_i64, _c_i64, _c_int, _vp, _vp, _vp, _c_dbl, _c_u64, _c_u64, _vp, _vp]),
    "dmo_cmaes_sample": (_c_int, [_vp, _vp, _vp, _c_int, _vp, _c_i64, _vp, _vp, _c_i64, _c_int, _vp]),
    "dmo_cmaes_update_cholesky": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_int, _c_dbl, _c_dbl, _c_dbl]),
    "dmo_gather_rows": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _vp]),
    "dmo_cmaes_generate": (_c_int, [_vp, _vp, _vp, _c_int, _vp, _c_i64, _vp, _vp, _c_i64, _c_int, _vp, _vp, _vp]),
    "dmo_cmaes_step_z": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_int, _vp]),
    "dmo_scale_rows": (_c_int, [_vp, _vp, _c_i64, _c_i64, _vp, _vp, _vp, _c_i64]),
    "dmo_benchmark_eval": (_c_int, [_vp, _c_int, _vp, _c_i64, _c_int, _c_int, _c_dbl, _vp]),
    "dmo_smpso_generate": (_c_int, [_vp, _vp, _vp, _c_int, _c_i64, _c_int, _vp, _vp, _vp, _c_dbl, _c_u64, _c_u64, _vp, _vp]),
    "dmo_smpso_update": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_int, _vp, _c_int, _c_i64, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
}

_lib = None
_ctx = None
_ctx_device = None
_lock = threading.Lock()


class DmoError(RuntimeError):
    pass


def load_library(path=None):
    """Load the shared library and declare every prototype.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise DmoError(
            f"dmosopt_b200: CUDA library {path} not found. Build it with `python -m dmosopt_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback."
        )
    lib = ctypes.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def default_device():
    for k in ("DMOSOPT_B200_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(k)
        if v is not None and v.strip() != "":
            return int(v)
    return 0


def context(device=None):
    """The process-wide context (one per process == one per GPU)."""
    global _ctx, _ctx_device
    with _lock:
        if _ctx is not None and (device is None or device == _ctx_device):
            return _ctx
        lib = load_library()
        dev = default_device() if device is None else int(device)
        h = _vp()
        st = lib.dmo_create(dev, ctypes.byref(h))
        if st != 0 or not h.value:
            raise DmoError(f"dmosopt_b200: dmo_create(device={dev}) failed with status {st}: no usable CUDA device (B200 required)")
        if _ctx is not None:
            lib.dmo_destroy(_ctx)
        _ctx, _ctx_device = h, dev
        return _ctx


def _check(st, what, ctx=None):
    if st != 0:
        msg = _lib.dmo_last_error(_ctx if ctx is None else ctx)
        raise DmoError(f"{what} failed (status {st}): {msg.decode() if msg else ''}")


# Additional contexts on the same GPU (own stream, own scratch): independent sub-problems of one call -- the swarms of an
# SMPSO update -- are issued from worker threads, one context each, so their latency-bound kernels (the rank chains)
# overlap on the device.  The C library is not re-entrant per context; different contexts may run concurrently.
_worker_ctx = []
_worker_pool = None


def worker_context(i):
    """The i-th worker context on the main context's GPU (created on first use)."""
    main = context()
    with _lock:
        while len(_worker_ctx) <= i:
            h = _vp()
            st = load_library().dmo_create(_ctx_device, ctypes.byref(h))
            if st != 0 or not h.value:
                raise DmoError(f"dmosopt_b200: dmo_create(device={_ctx_device}) failed for a worker context (status {st})")
            _worker_ctx.append(h)
    assert main is not None
    return _worker_ctx[i]


def worker_pool():
    global _worker_pool
    if _worker_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _worker_pool = ThreadPoolExecutor(max_workers=8, thread_name_prefix="dmosopt_b200_worker")
    return _worker_pool


def _ptr(a):
    """Raw pointer of a NumPy array, a torch CUDA tensor (data_ptr) or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return int(a.data_ptr())
    if isinstance(a, int):
        return a
    raise TypeError(f"cannot pass {type(a)} to the CUDA library")


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


# --------------------------------------------------------------------------- context utilities
def synchronize():
    _check(load_library().dmo_synchronize(context()), "dmo_synchronize")


def stream_ptr():
    """The CUDA stream (cudaStream_t as an integer) every library call is issued on: wrap it with
    ``torch.cuda.ExternalStream`` to order torch / NCCL work with the library without device-wide synchronisation."""
    return int(load_library().dmo_stream(context()))


def launch_count():
    lib = load_library()
    return int(lib.dmo_launch_count(context())) + sum(int(lib.dmo_launch_count(c)) for c in _worker_ctx)


def sm_count():
    return int(load_library().dmo_sm_count(context()))


def timer_begin():
    _check(load_library().dmo_timer_begin(context()), "dmo_timer_begin")


def timer_end():
    ms = ctypes.c_float()
    _check(load_library().dmo_timer_end(context(), ctypes.byref(ms)), "dmo_timer_end")
    return float(ms.value)


def flush_l2():
    _check(load_library().dmo_flush_l2(context()), "dmo_flush_l2")


def transfer_bytes():
    h2d = d2h = 0
    for c in [context()] + list(_worker_ctx):
        a, b = _c_u64(0), _c_u64(0)
        _check(load_library().dmo_transfer_bytes(c, ctypes.byref(a), ctypes.byref(b)), "dmo_transfer_bytes")
        h2d, d2h = h2d + int(a.value), d2h + int(b.value)
    return h2d, d2h


def profile_enable(on=True):
    _check(load_library().dmo_profile_enable(context(), 1 if on else 0), "dmo_profile_enable")


def profile_report():
    """{kernel name: (total ms, launches)} recorded since profile_enable(True)."""
    buf = ctypes.create_string_buffer(1 << 16)
    _check(load_library().dmo_profile_report(context(), buf, len(buf)), "dmo_profile_report")
    out = {}
    for line in buf.value.decode().splitlines():
        name, ms, cnt = line.rsplit(" ", 2)
        out[name] = (float(ms), int(cnt))
    return out


def round_f32(dev_ptr, n):
    _check(load_library().dmo_round_f32(context(), _ptr(dev_ptr), int(n)), "dmo_round_f32")


class DeviceArray:
    """A typed device buffer owned by the library context (for callers that keep populations resident)."""

    def __init__(self, shape, dtype=np.float64):
        self.shape = tuple(np.atleast_1d(shape).tolist()) if not isinstance(shape, tuple) else shape
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = _vp()
        _check(load_library().dmo_device_alloc(context(), ctypes.byref(p), max(self.nbytes, 1)), "dmo_device_alloc")
        self.ptr = p.value

    def data_ptr(self):
        return self.ptr

    def offset(self, nelem):
        """Raw pointer ``nelem`` elements into the buffer."""
        return self.ptr + int(nelem) * self.dtype.itemsize

    def upload(self, a):
        a = np.ascontiguousarray(a, dtype=self.dtype)
        assert a.nbytes <= self.nbytes
        _check(load_library().dmo_memcpy(context(), self.ptr, a.ctypes.data, a.nbytes), "dmo_memcpy")
        return self

    def download(self, count=None):
        n = int(np.prod(self.shape)) if count is None else int(count)
        out = np.empty(n, dtype=self.dtype)
        _check(load_library().dmo_memcpy(context(), out.ctypes.data, self.ptr, out.nbytes), "dmo_memcpy")
        return out.reshape(self.shape) if count is None else out

    def free(self):
        if self.ptr:
            load_library().dmo_device_free(context(), self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def memcpy(dst, src, nbytes):
    _check(load_library().dmo_memcpy(context(), _ptr(dst), _ptr(src), int(nbytes)), "dmo_memcpy")


# Page-locked host buffers are pooled: cudaHostAlloc of a population-sized block costs milliseconds, and the plugins
# hand out one offspring matrix per generation.  A block returns to the pool when the last NumPy view of it dies.
_pin_pool = {}
_pin_pool_bytes = 0
_PIN_POOL_LIMIT = 1 << 30
# page-locked bytes currently handed out (not pooled).  Callers such as MOASMO.optimize keep every offspring matrix of
# an epoch alive (x_new history): beyond this budget new offspring matrices are ordinary pageable arrays.
_pin_live_bytes = 0
_PIN_LIVE_LIMIT = int(os.environ.get("DMOSOPT_B200_PINNED_LIMIT", str(4 << 30)))
# Device mirrors of read-only host arrays the library itself produced (offspring matrix, population state):
# {host address: (nbytes, DeviceArray)}.  ``_in`` substitutes the device address, so data that was born on the GPU is
# not shipped back over PCIe when the caller hands it to the next call.  Only non-writeable arrays qualify: a
# caller who wants to edit must copy, and the copy has no mirror.
_mirrors = {}


def _pin_release(ptr, nbytes):
    global _pin_pool_bytes, _pin_live_bytes
    _pin_live_bytes -= nbytes
    _mirrors.pop(ptr, None)
    lst = _pin_pool.setdefault(nbytes, [])
    if len(lst) < 4 and _pin_pool_bytes + nbytes <= _PIN_POOL_LIMIT:
        lst.append(ptr)
        _pin_pool_bytes += nbytes
    elif _lib is not None:
        _lib.dmo_host_free(ptr)


def pinned_empty(shape, dtype=np.float64):
    """NumPy array backed by page-locked host memory (pooled; recycled when the last view is collected)."""
    global _pin_pool_bytes, _pin_live_bytes
    import weakref

    lib = load_library()
    context()
    dt = np.dtype(dtype)
    count = int(np.prod(shape))
    nbytes = (max(count * dt.itemsize, 1) + 4095) & ~4095
    lst = _pin_pool.get(nbytes)
    if lst:
        addr = lst.pop()
        _pin_pool_bytes -= nbytes
    else:
        p = _vp()
        if lib.dmo_host_alloc(ctypes.byref(p), nbytes) != 0:
            raise DmoError("dmo_host_alloc failed")
        addr = p.value
    buf = (ctypes.c_char * nbytes).from_address(addr)
    _pin_live_bytes += nbytes
    weakref.finalize(buf, _pin_release, addr, nbytes)
    return np.frombuffer(buf, dtype=dt, count=count).reshape(shape)


def mirror_register(host, dev):
    """Declare ``dev`` (DeviceArray) the device copy of the pinned array ``host`` (from pinned_empty)."""
    _mirrors[host.ctypes.data] = (host.nbytes, dev)


def mirror_drop(a):
    """Forget (and free) the device copy of ``a``: the host array stays valid, later uses simply upload it again.

    The optimizers call this once ``update`` has consumed an offspring matrix, so a caller that keeps every x_gen of an
    epoch (MOASMO.optimize's history) holds host memory only, not one HBM buffer per generation."""
    if not isinstance(a, np.ndarray):
        return
    addr = a.ctypes.data
    ent = _mirrors.get(addr)
    if ent is None:
        for base, (nbytes, dev) in list(_mirrors.items()):
            if base <= addr < base + nbytes:
                addr, ent = base, (nbytes, dev)
                break
    if ent is not None:
        _mirrors.pop(addr, None)
        ent[1].free()


def mirror_upload(host):
    """Refresh the device mirror of ``host`` after a host-side write through its writable base."""
    ent = _mirrors.get(host.ctypes.data)
    if ent is not None:
        ent[1].upload(host)


def mirror_ptr(a, require_readonly=True):
    """Device address mirroring the host array ``a`` (or an interior C-contiguous view of it), else None."""
    if not _mirrors or not isinstance(a, np.ndarray) or not a.flags.c_contiguous:
        return None
    if require_readonly and a.flags.writeable:
        return None
    addr = a.ctypes.data
    ent = _mirrors.get(addr)
    if ent is not None:
        return ent[1].ptr if a.nbytes <= ent[0] and ent[1].ptr else None
    for base, (nbytes, dev) in list(_mirrors.items()):  # a finaliser may drop an entry while we look
        if base <= addr and addr + a.nbytes <= base + nbytes and dev.ptr:
            return dev.ptr + (addr - base)
    return None


def _in(a):
    """Pointer for an input array: the device mirror when the library holds one, else the host address."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        m = mirror_ptr(a)
        return m if m is not None else a.ctypes.data
    return _ptr(a)


def mirrored_readonly(a):
    """(read-only view, writable pinned base) of a page-locked, device-mirrored copy of ``a``.

    Returns (copy of a, None) when no CUDA context can be created (host-only unit tests)."""
    a = np.asarray(a)
    try:
        base = pinned_empty(a.shape, a.dtype)
        base[...] = a
        dev = DeviceArray(a.shape, a.dtype).upload(base)
    except DmoError:
        return np.array(a, copy=True), None
    mirror_register(base, dev)
    view = base.view()
    view.flags.writeable = False
    return view, base


def copy_into_pooled(a):
    """Writable copy of ``a`` in a pooled page-locked buffer; a plain ``a.copy()`` when no CUDA context exists."""
    a = np.asarray(a)
    if a.nbytes < (1 << 20):
        return a.copy()
    try:
        out = pinned_empty(a.shape, a.dtype)
    except DmoError:
        return a.copy()
    m = mirror_ptr(a)
    if m is not None:  # the DMA engine copies device -> pinned host faster than one host thread copies host -> host
        memcpy(out, m, a.nbytes)
    else:
        np.copyto(out, a)
    return out


def pinned_like(a):
    """Page-locked copy of ``a`` (same dtype / values); falls back to a plain copy when no context exists yet."""
    a = np.asarray(a)
    try:
        out = pinned_empty(a.shape, a.dtype)
    except DmoError:
        return np.array(a, copy=True)
    out[...] = a
    return out


# --------------------------------------------------------------------------- A1/A2
def rank_nd(Y):
    """dda.dda_ens (dmosopt/dda.py:97-152) -> int64 rank array (canonical non-dominated rank)."""
    Y = _f64(Y)
    n, M = Y.shape
    rank = np.empty(n, dtype=np.int32)
    _check(load_library().dmo_rank_nd(context(), _ptr(Y), n, M, _ptr(rank)), "dmo_rank_nd")
    return rank.astype(np.intp)


# --------------------------------------------------------------------------- A3/A4
def crowding_distance(Y):
    Y = _f64(Y)
    n, M = Y.shape
    D = np.empty(n, dtype=np.float64)
    _check(load_library().dmo_crowding_distance(context(), _ptr(Y), n, M, _ptr(D)), "dmo_crowding_distance")
    return D


def euclidean_distance(Y):
    Y = _f64(Y)
    n, M = Y.shape
    D = np.empty(n, dtype=np.float64)
    _check(load_library().dmo_euclidean_distance(context(), _ptr(Y), n, M, _ptr(D)), "dmo_euclidean_distance")
    return D


# --------------------------------------------------------------------------- A5
def _extra_keys(extra):
    if not extra:
        return None, 0, []
    arrs = [_f64(e) for e in extra]
    tab = (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
    return ctypes.cast(tab, ctypes.c_void_p), len(arrs), arrs


def order_mo(Y, metric=METRIC_NONE, extra_desc_keys=None):
    """(perm, rank[perm], dist[perm] or None): the ordering of MOEA.orderMO (dmosopt/MOEA.py:300-347)."""
    Y = _f64(Y)
    n, M = Y.shape
    perm = np.empty(n, dtype=np.int64)
    rank = np.empty(n, dtype=np.int32)
    dist = np.empty(n, dtype=np.float64) if metric != METRIC_NONE else None
    tab, nex, keep = _extra_keys(extra_desc_keys)
    _check(load_library().dmo_order_mo(context(), _ptr(Y), n, M, metric, tab, nex, _ptr(perm), _ptr(rank), _ptr(dist)), "dmo_order_mo")
    return perm, rank.astype(np.intp), dist


def remove_worst(X, Y, keep, metric=METRIC_NONE, extra_desc_keys=None):
    """First ``keep`` rows of the sortMO order (dmosopt/MOEA.py:398-423): (X, Y, rank, perm)."""
    X = _f64(X)
    Y = _f64(Y)
    n, d = X.shape
    M = Y.shape[1]
    keep = int(min(keep, n))
    Xo = np.empty((keep, d), dtype=np.float64)
    Yo = np.empty((keep, M), dtype=np.float64)
    rank = np.empty(keep, dtype=np.int32)
    perm = np.empty(keep, dtype=np.int64)
    tab, nex, hold = _extra_keys(extra_desc_keys)
    _check(
        load_library().dmo_remove_worst(context(), _ptr(X), _ptr(Y), n, d, M, metric, tab, nex, keep, _ptr(Xo), _ptr(Yo), _ptr(rank), _ptr(perm)),
        "dmo_remove_worst",
    )
    return Xo, Yo, rank.astype(np.intp), perm


def remove_worst_pair(Xa, Ya, Xb, Yb, keep, metric=METRIC_NONE, out_X=None):
    """remove_worst(vstack(Xa, Xb), vstack(Ya, Yb), keep) without the host-side concatenation.

    ``out_X`` (optional, float64 C-contiguous (keep, d)) receives the surviving rows directly; it may be the writable
    base of ``Xb``.  When ``out_X`` has a device mirror the survivors are written to the mirror and copied out once.
    """
    Xa, Ya, Xb, Yb = _f64(Xa), _f64(Ya), _f64(Xb), _f64(Yb)
    na, d = Xa.shape
    nb = Xb.shape[0]
    M = Ya.shape[1]
    keep = int(min(keep, na + nb))
    if out_X is not None and (out_X.dtype != np.float64 or not out_X.flags.c_contiguous or out_X.shape != (keep, d)):
        out_X = None
    Xo = out_X if out_X is not None else pinned_empty((keep, d), np.float64)
    Yo = np.empty((keep, M), dtype=np.float64)
    rank = np.empty(keep, dtype=np.int32)
    perm = np.empty(keep, dtype=np.int64)
    xo_dev = mirror_ptr(Xo, require_readonly=False) if out_X is not None else None
    _check(
        load_library().dmo_remove_worst_pair(context(), _in(Xa), _in(Ya), na, _in(Xb), _in(Yb), nb, d, M, metric, keep,
                                             xo_dev if xo_dev is not None else _ptr(Xo), _ptr(Yo), _ptr(rank), _ptr(perm)),
        "dmo_remove_worst_pair",
    )
    if xo_dev is not None:
        memcpy(Xo, xo_dev, Xo.nbytes)
    return Xo, Yo, rank.astype(np.intp), perm


# --------------------------------------------------------------------------- A6
def tournament(rank, poolsize, seed, stream_id, crowd=None, return_uniforms=False):
    rank = np.ascontiguousarray(rank, dtype=np.int32)
    pop = rank.shape[0]
    cr = None if crowd is None else _f64(crowd)
    pool = np.empty(int(poolsize), dtype=np.int64)
    u = np.empty(pop, dtype=np.float64) if return_uniforms else None
    _check(
        load_library().dmo_tournament(context(), _ptr(rank), _ptr(cr), pop, int(poolsize), int(seed) & (2**64 - 1), int(stream_id), _ptr(pool), _ptr(u)),
        "dmo_tournament",
    )
    return (pool, u) if return_uniforms else pool


# --------------------------------------------------------------------------- A7/A8
def mutation_u(parents, u, di_mutation, xlb, xub, mutation_rate):
    parents = np.atleast_2d(_f64(parents))
    u = np.atleast_2d(_f64(u))
    n, d = parents.shape
    di = _f64(np.broadcast_to(np.asarray(di_mutation, dtype=np.float64), (d,)))
    out = np.empty((n, d), dtype=np.float64)
    lb, ub = _f64(xlb), _f64(xub)  # named: the arrays must outlive the call
    _check(load_library().dmo_mutation_u(context(), _ptr(parents), _ptr(u), n, d, _ptr(di), _ptr(lb), _ptr(ub), float(mutation_rate), _ptr(out)), "dmo_mutation_u")
    return out


def sbx_u(parent1, parent2, u, di_crossover, xlb, xub):
    p1 = np.atleast_2d(_f64(parent1))
    p2 = np.atleast_2d(_f64(parent2))
    u = np.atleast_2d(_f64(u))
    n, d = p1.shape
    di = _f64(np.broadcast_to(np.asarray(di_crossover, dtype=np.float64), (d,)))
    c1 = np.empty((n, d), dtype=np.float64)
    c2 = np.empty((n, d), dtype=np.float64)
    lb, ub = _f64(xlb), _f64(xub)
    _check(load_library().dmo_sbx_u(context(), _ptr(p1), _ptr(p2), _ptr(u), n, d, _ptr(di), _ptr(lb), _ptr(ub), _ptr(c1), _ptr(c2)), "dmo_sbx_u")
    return c1, c2


# --------------------------------------------------------------------------- A9
def nsga2_generate(pop_x, pool_idx, popsize, crossover_prob, mutation_prob, mutation_rate, di_crossover, di_mutation, xlb, xub, seed, stream_id, return_draws=False):
    """Offspring of the NSGA-II / AGE-MOEA variation loop (dmosopt/NSGA2.py:142-178).

    Returns (x_gen (P, d), child_kind (P,) int32 [0/1 = SBX child 1/2, 2 = mutant][, draws]).
    ``draws`` (if requested) is a dict with the random draws the kernel used, for replay on the
    CPU oracle: u_cross (T,), u_mut (T,), pair (T, 2), single (T,), u_genes (T, 2, d), T = dmo_nsga2_plan_length
    (2*popsize+64 for the default rates).
    """
    pop_x = _f64(pop_x)
    npop, d = pop_x.shape
    pool_idx = np.ascontiguousarray(pool_idx, dtype=np.int64)
    popsize = int(popsize)
    T = int(load_library().dmo_nsga2_plan_length(popsize, float(crossover_prob), float(mutation_prob)))
    if T <= 0:
        raise DmoError("nsga2_generate: crossover_prob / mutation_prob too small to plan the variation loop")
    # the offspring matrix stays on the device as the mirror of the (read-only, page-locked) array handed back
    x_dev = DeviceArray((popsize + 1, d), np.float64)
    kind = np.empty(popsize + 1, dtype=np.int32)
    nch = np.zeros(1, dtype=np.int64)
    draws = np.empty(T * (5 + 2 * d), dtype=np.float64) if return_draws else None
    dic = _f64(np.broadcast_to(np.asarray(di_crossover, dtype=np.float64), (d,)))
    dim = _f64(np.broadcast_to(np.asarray(di_mutation, dtype=np.float64), (d,)))
    lb, ub = _f64(xlb), _f64(xub)
    _check(
        load_library().dmo_nsga2_generate(
            context(), _in(pop_x), npop, d, _ptr(pool_idx), pool_idx.shape[0], popsize, float(crossover_prob), float(mutation_prob),
            float(mutation_rate), _ptr(dic), _ptr(dim), _ptr(lb), _ptr(ub), int(seed) & (2**64 - 1), int(stream_id),
            x_dev.ptr, _ptr(kind), _ptr(nch), _ptr(draws),
        ),
        "dmo_nsga2_generate",
    )
    P = int(nch[0])
    if _pin_live_bytes < _PIN_LIVE_LIMIT:
        x_gen = pinned_empty((popsize + 1, d), np.float64)
    else:  # the caller is hoarding offspring matrices: pageable memory from here on (mirror dropped with the array)
        import weakref

        x_gen = np.empty((popsize + 1, d), dtype=np.float64)
        weakref.finalize(x_gen, _mirrors.pop, x_gen.ctypes.data, None)
    if P:
        memcpy(x_gen, x_dev.ptr, P * d * 8)
    mirror_register(x_gen, x_dev)
    x_gen.flags.writeable = False
    if not return_draws:
        return x_gen[:P], kind[:P]
    dd = {
        "u_cross": draws[0:T],
        "u_mut": draws[T : 2 * T],
        "pair": draws[2 * T : 4 * T].reshape(T, 2).astype(np.int64),
        "single": draws[4 * T : 5 * T].astype(np.int64),
        "u_genes": draws[5 * T :].reshape(T, 2, d),
    }
    return x_gen[:P], kind[:P], dd


# --------------------------------------------------------------------------- N1: exact-GP fit for given hyper-parameters
def gp_fit(X_train, y, constant, length_scale, noise, kernel=KERNEL_MATERN52, jitter=1e-10, want_L=True, want_alpha=True):
    """(L (M,N,N) or None, alpha (M,N) or None, lml (M,)) of the exact GP with the given hyper-parameters, per objective:
    K = c k(X, X) + (noise + jitter) I, L = chol(K), alpha = K^-1 y, lml = log marginal likelihood (dmo_gp_fit).
    X_train (N,d) normalised inputs, y (M,N) normalised targets, length_scale (M,d)."""
    X_train = _f64(X_train)
    N, d = X_train.shape
    y = _f64(y)
    M = y.shape[0]
    ls = np.empty((M, d), dtype=np.float64)
    for m in range(M):
        ls[m, :] = np.asarray(length_scale[m], dtype=np.float64)
    cst, nz = _f64(constant), _f64(noise)
    assert y.shape == (M, N) and cst.shape == (M,) and nz.shape == (M,)
    L = np.empty((M, N, N), dtype=np.float64) if want_L else None
    alpha = np.empty((M, N), dtype=np.float64) if want_alpha else None
    lml = np.empty(M, dtype=np.float64)
    _check(load_library().dmo_gp_fit(context(), N, d, M, int(kernel), _ptr(X_train), _ptr(y), _ptr(cst), _ptr(ls), _ptr(nz), float(jitter), _ptr(L), _ptr(alpha),
                                     _ptr(lml)), "dmo_gp_fit")
    return L, alpha, lml


# --------------------------------------------------------------------------- A18
class GPHandle:
    """Owns a dmo_gp object (posterior state resident in HBM)."""

    def __init__(self, X_train, alpha, factor, constant, length_scale, noise, y_mean, y_std, xlb, xub, kernel=KERNEL_MATERN52, factor_is_inverse=False):
        lib = load_library()
        X_train = _f64(X_train)
        N, d = X_train.shape
        alpha = _f64(alpha)
        M = alpha.shape[0]
        factor = _f64(factor)
        assert factor.shape == (M, N, N), factor.shape
        ls = np.empty((M, d), dtype=np.float64)
        for m in range(M):
            ls[m, :] = np.asarray(length_scale[m], dtype=np.float64)
        self.N, self.d, self.M = N, d, M
        cst, nz, ym, ys, lb, ub = _f64(constant), _f64(noise), _f64(y_mean), _f64(y_std), _f64(xlb), _f64(xub)
        assert cst.shape == (M,) and nz.shape == (M,) and ym.shape == (M,) and ys.shape == (M,) and lb.shape == (d,) and ub.shape == (d,)
        h = _vp()
        _check(
            lib.dmo_gp_create(
                context(), N, d, M, int(kernel), _ptr(X_train), _ptr(alpha), _ptr(factor), 1 if factor_is_inverse else 0, _ptr(cst),
                _ptr(ls), _ptr(nz), _ptr(ym), _ptr(ys), _ptr(lb), _ptr(ub), ctypes.byref(h),
            ),
            "dmo_gp_create",
        )
        self._h = h

    def set_linear_mean(self, weight, bias):
        """Prior mean w_m . x_n + b_m per objective (gpytorch LinearMean, A19); ``None, None`` removes it."""
        if weight is None and bias is None:
            _check(load_library().dmo_gp_set_linear_mean(context(), self._h, None, None), "dmo_gp_set_linear_mean")
            return
        w = _f64(np.asarray(weight, dtype=np.float64).reshape(self.M, self.d))
        b = _f64(np.asarray(bias, dtype=np.float64).reshape(self.M))
        _check(load_library().dmo_gp_set_linear_mean(context(), self._h, _ptr(w), _ptr(b)), "dmo_gp_set_linear_mean")

    def predict(self, X, return_var=True, precision=GP_FP64):
        X = _f64(X)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        P = X.shape[0]
        mean = pinned_empty((P, self.M), np.float64)
        var = pinned_empty((P, self.M), np.float64) if return_var else None
        _check(load_library().dmo_gp_predict(context(), self._h, _in(X), P, _ptr(mean), _ptr(var), int(precision)), "dmo_gp_predict")
        return mean, var

    def auto_info(self):
        """What precision=GP_AUTO does for this model (runs the one-off calibration if needed)."""
        mt, vt, rows = _c_int(0), _c_int(0), _c_i64(0)
        em, ev, th = _c_dbl(0.0), _c_dbl(0.0), _c_dbl(0.0)
        _check(load_library().dmo_gp_auto_info(context(), self._h, ctypes.byref(mt), ctypes.byref(vt), ctypes.byref(em), ctypes.byref(ev),
                                               ctypes.byref(th), ctypes.byref(rows)), "dmo_gp_auto_info")
        # mean_from_contraction is always False (bit 1 is reserved); the key stays so that the dict, which bench.py
        # records as gp_auto, keeps its shape
        return {"mean_tensor": bool(mt.value & 1), "mean_from_contraction": bool(mt.value & 2), "mean_only_tensor": bool(mt.value & 4),
                "var_tensor": bool(vt.value), "mean_err": em.value,
                "var_err": ev.value, "theta": th.value, "last_refined": int(rows.value)}

    def close(self):
        if getattr(self, "_h", None) is not None and _lib is not None and _ctx is not None:
            _lib.dmo_gp_destroy(_ctx, self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# --------------------------------------------------------------------------- A16/A17
def hypervolume(F, ref, rank=None):
    """Exact hypervolume; ``rank`` (optional): non-dominated ranks of the rows within the superset they were selected from
    by rank (skips the non-dominated filter, see dmo_hypervolume_ranked)."""
    F = _f64(F)
    if F.ndim == 1:
        F = F.reshape(1, -1)
    n, M = F.shape
    ref = _f64(ref)
    out = _c_dbl(0.0)
    if rank is None:
        _check(load_library().dmo_hypervolume(context(), _ptr(F), n, M, _ptr(ref), ctypes.byref(out)), "dmo_hypervolume")
    else:
        rk = np.ascontiguousarray(rank, dtype=np.int32)
        assert rk.shape == (n,)
        _check(load_library().dmo_hypervolume_ranked(context(), _ptr(F), n, M, _ptr(ref), _ptr(rk), ctypes.byref(out)), "dmo_hypervolume_ranked")
    return float(out.value)


def ehvi_select(F, means, variances, ref, k, nds=True, return_scores=False):
    F = _f64(F)
    means = _f64(means)
    variances = _f64(variances)
    nf, M = F.shape
    nc = means.shape[0]
    k = int(min(k, nc))
    sel = np.empty(k, dtype=np.int64)
    score = np.empty(nc, dtype=np.float64) if return_scores else None
    ref = _f64(ref)
    _check(
        load_library().dmo_ehvi_select(context(), _ptr(F), nf, _ptr(means), _ptr(variances), nc, M, _ptr(ref), 1 if nds else 0, k, _ptr(sel), _ptr(score)),
        "dmo_ehvi_select",
    )
    return (sel, score) if return_scores else sel


# --------------------------------------------------------------------------- A21
def get_duplicates(X, eps=1e-16, Y=None):
    X = _f64(X)
    n, d = X.shape
    out = np.empty(n, dtype=np.uint8)
    if Y is None:
        _check(load_library().dmo_get_duplicates(context(), _in(X), n, d, float(eps), _ptr(out)), "dmo_get_duplicates")
    else:
        Y = _f64(Y)
        assert Y.ndim == 2 and Y.shape[1] == d, (X.shape, Y.shape)
        _check(load_library().dmo_get_duplicates_pair(context(), _in(X), n, _in(Y), Y.shape[0], d, float(eps), _ptr(out)), "dmo_get_duplicates_pair")
    return out.astype(bool)


# --------------------------------------------------------------------------- A11 AGE-MOEA
def age_survival(yn, nn, p, extreme):
    """Greedy part of AGEMOEA.survival_score (dmosopt/AGEMOEA.py:398-428) -> crowding values (m,)."""
    yn = _f64(yn)
    nn = _f64(nn)
    m, M = yn.shape
    ext = np.ascontiguousarray(extreme, dtype=np.int32)
    crowd = np.empty(m, dtype=np.float64)
    _check(load_library().dmo_age_survival(context(), _ptr(yn), _ptr(nn), m, M, float(p), _ptr(ext), ext.shape[0], _ptr(crowd)), "dmo_age_survival")
    return crowd


# --------------------------------------------------------------------------- A12 SMPSO
def smpso_velocity(position, velocity, leader1, leader2, w, c1, r1, c2, r2, chi, xlb, xub):
    f32_diff = 1 if (np.asarray(leader1).dtype == np.float32 and np.asarray(position).dtype == np.float32) else 0
    pos = np.ascontiguousarray(position, dtype=np.float32)
    vel = _f64(velocity)
    l1 = _f64(leader1)
    l2 = _f64(leader2)
    n, d = pos.shape
    lb, ub = _f64(xlb), _f64(xub)
    out = np.empty((n, d), dtype=np.float64)
    _check(
        load_library().dmo_smpso_velocity(context(), _ptr(pos), _ptr(vel), _ptr(l1), _ptr(l2), f32_diff, n, d, float(w), float(c1), float(r1), float(c2), float(r2),
                                          float(chi), _ptr(lb), _ptr(ub), _ptr(out)),
        "dmo_smpso_velocity",
    )
    return out


def mutate_groups(pop_x, group_size, n_groups, per_group, di_mutation, xlb, xub, mutation_rate, seed, stream_id, return_parents=False):
    pop_x = _f64(pop_x)
    d = pop_x.shape[1]
    total = int(n_groups) * int(per_group)
    di = _f64(np.broadcast_to(np.asarray(di_mutation, dtype=np.float64), (d,)))
    lb, ub = _f64(xlb), _f64(xub)
    out = np.empty((total, d), dtype=np.float64)
    par = np.empty(total, dtype=np.int64) if return_parents else None
    _check(
        load_library().dmo_mutate_groups(context(), _ptr(pop_x), int(group_size), int(n_groups), int(per_group), d, _ptr(di), _ptr(lb), _ptr(ub),
                                         float(mutation_rate), int(seed) & (2**64 - 1), int(stream_id), _ptr(out), _ptr(par)),
        "dmo_mutate_groups",
    )
    return (out, par) if return_parents else out


BENCHMARKS = {"zdt1": 0, "zdt3": 1, "dtlz1": 10, "dtlz2": 11, "dtlz3": 12, "dtlz4": 13, "dtlz5": 14, "dtlz7": 16, "wfg4": 24}


def benchmark_eval(name, X, n_obj, alpha=100.0):
    """Rows of X through one of the reference's benchmark functions (dmosopt/benchmarks/moo_benchmarks.py), on the GPU."""
    X = _f64(X)
    n, d = X.shape
    Y = np.empty((n, int(n_obj)), dtype=np.float64)
    _check(load_library().dmo_benchmark_eval(context(), BENCHMARKS[name], _in(X), n, d, int(n_obj), float(alpha), _ptr(Y)), "dmo_benchmark_eval")
    return Y


class SmpsoSwarms:
    """The swarm state of SMPSO resident in HBM (dmo_smpso_generate / dmo_smpso_update, csrc/smpso.cu): positions and
    objectives as float64 arrays holding float32-representable values, velocities in float64."""

    def __init__(self, parm, obj, vel, swarms, pop):
        parm, obj, vel = np.asarray(parm), np.asarray(obj), np.asarray(vel)
        self.swarms, self.pop, self.d, self.M = int(swarms), int(pop), parm.shape[1], obj.shape[1]
        n = self.swarms * self.pop
        assert parm.shape[0] == n and obj.shape[0] == n and vel.shape == (n, self.d)
        self.parm = DeviceArray((n, self.d)).upload(_f64(parm))
        self.obj = DeviceArray((n, self.M)).upload(_f64(obj))
        self.vel = DeviceArray((n, self.d)).upload(_f64(vel))

    def generate(self, di_mutation, xlb, xub, mutation_rate, seed, stream_id):
        """x_gen (2 * swarms * pop, d), laid out as SMPSO.py:163-184 does: the reference's float32 values, handed out as the
        float64 array MOEA.generate turns them into (np.clip against float64 bounds, MOEA.py:155) -- read-only, page-locked,
        with its device copy kept as a mirror so that evaluate(x_gen) / update(x_gen, ...) do not ship it back over PCIe."""
        di = _f64(np.broadcast_to(np.asarray(di_mutation, dtype=np.float64), (self.d,)))
        lb, ub = _f64(xlb), _f64(xub)
        rows = 2 * self.swarms * self.pop
        x_dev = DeviceArray((rows, self.d), np.float64)
        _check(load_library().dmo_smpso_generate(context(), self.parm.ptr, self.vel.ptr, self.swarms, self.pop, self.d, _ptr(di), _ptr(lb), _ptr(ub),
                                                 float(mutation_rate), int(seed) & (2**64 - 1), int(stream_id), None, x_dev.ptr), "dmo_smpso_generate")
        out = pinned_empty((rows, self.d), np.float64)
        memcpy(out, x_dev.ptr, out.nbytes)
        mirror_register(out, x_dev)
        out.flags.writeable = False
        return out

    def update(self, x_gen, y_gen, scalars, xlb, xub, metric, parm_out, obj_out):
        """One update_strategy (SMPSO.py:187-238) on the resident state; writes the new float32 state into parm_out /
        obj_out and returns (ranks (swarms, pop) intp, perm (swarms, pop) int64)."""
        n = self.swarms * self.pop
        x_gen = np.asarray(x_gen)
        if x_gen.dtype == np.float32:
            xg, is32 = np.ascontiguousarray(x_gen[:n]), 1
        else:
            xg, is32 = _f64(x_gen[:n]), 0  # a view of the caller's array: its device mirror (if any) is found by address
        yg = _f64(np.asarray(y_gen)[:n])
        sc = _f64(scalars)
        assert sc.shape == (self.swarms, 8) and xg.shape == (n, self.d) and yg.shape == (n, self.M)
        lb, ub = _f64(xlb), _f64(xub)
        ranks = np.empty(n, dtype=np.int32)
        perm = np.empty(n, dtype=np.int64)
        po = parm_out if (parm_out.dtype == np.float32 and parm_out.flags.c_contiguous) else np.empty((n, self.d), np.float32)
        oo = obj_out if (obj_out.dtype == np.float32 and obj_out.flags.c_contiguous) else np.empty((n, self.M), np.float32)
        lib = load_library()
        if self.swarms > 1 and os.environ.get("DMOSOPT_B200_SMPSO_THREADS", "1") != "0":
            # the swarms are independent (SMPSO.py:211-228): one worker context and thread per swarm, so the per-swarm
            # rank chains (latency bound, a fraction of the SMs each) overlap on the device
            synchronize()  # state and inputs produced on the main context's stream are complete
            pxg, pyg, psc, prk, ppm, ppo, poo = _in(xg), _in(yg), _ptr(sc), _ptr(ranks), _ptr(perm), _ptr(po), _ptr(oo)
            plb, pub = _ptr(lb), _ptr(ub)
            xsz = 4 if is32 else 8
            pop, d, M = self.pop, self.d, self.M

            def one(p):
                ctx, off = worker_context(p), p * pop
                st = lib.dmo_smpso_update(ctx, self.parm.ptr + off * d * 8, self.obj.ptr + off * M * 8, self.vel.ptr + off * d * 8, pxg + off * d * xsz, is32,
                                          pyg + off * M * 8, 1, pop, d, M, int(metric), psc + p * 64, plb, pub, prk + off * 4, ppm + off * 8,
                                          ppo + off * d * 4, poo + off * M * 4)
                return st, ctx

            for st, ctx in list(worker_pool().map(one, range(self.swarms))):
                _check(st, "dmo_smpso_update", ctx)
        else:
            _check(lib.dmo_smpso_update(context(), self.parm.ptr, self.obj.ptr, self.vel.ptr, _in(xg), is32, _in(yg), self.swarms, self.pop, self.d,
                                        self.M, int(metric), _ptr(sc), _ptr(lb), _ptr(ub), _ptr(ranks), _ptr(perm), _ptr(po), _ptr(oo)), "dmo_smpso_update")
        if po is not parm_out:
            parm_out[...] = po
        if oo is not obj_out:
            obj_out[...] = oo
        return ranks.astype(np.intp).reshape(self.swarms, self.pop), perm.reshape(self.swarms, self.pop)

    def velocity_into(self, out):
        """Copy the resident velocities into ``out`` (float64, C-contiguous; page-locked state arrays take the DMA path)."""
        if out.dtype == np.float64 and out.flags.c_contiguous:
            memcpy(out, self.vel.ptr, out.nbytes)
        else:
            out[...] = self.vel.download()


# --------------------------------------------------------------------------- device-resident per-individual state
class ResidentRows:
    """(n, ...) float64 array that lives in HBM across generations (MO-CMA-ES keeps one (d, d) Cholesky factor, its
    inverse and one evolution path per parent: 604 MB at pop 131 072, d = 24).  NumPy sees it through ``__array__`` /
    indexing (a device -> host copy on demand), the kernels through ``ptr``."""

    def __init__(self, dev, shape):
        self.dev = dev
        self.shape = tuple(int(v) for v in shape)
        self.dtype = np.dtype(np.float64)
        self.ndim = len(self.shape)

    @property
    def ptr(self):
        return self.dev.ptr

    def data_ptr(self):
        return self.dev.ptr

    @property
    def row_elems(self):
        return int(np.prod(self.shape[1:])) if len(self.shape) > 1 else 1

    def __len__(self):
        return self.shape[0]

    def __array__(self, dtype=None, copy=None):
        n = int(np.prod(self.shape))
        a = self.dev.download(n).reshape(self.shape) if n else np.zeros(self.shape)
        return a if dtype is None else a.astype(dtype)

    def __getitem__(self, key):
        return np.asarray(self)[key]

    def copy(self):
        return gather_rows(self, np.arange(self.shape[0], dtype=np.int64))


def resident_rows(a):
    """Upload a host array as a ResidentRows (no-op for one)."""
    if isinstance(a, ResidentRows):
        return a
    a = _f64(a)
    return ResidentRows(DeviceArray(a.shape, np.float64).upload(a), a.shape)


def gather_rows(src, idx, alt=None, sel=None):
    """ResidentRows with rows ``(alt if sel[i] else src)[idx[i]]`` (dmo_gather_rows): device -> device."""
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    n = idx.shape[0]
    shape = (n,) + src.shape[1:]
    out = ResidentRows(DeviceArray(shape, np.float64), shape)
    if n == 0:
        return out
    sl = None if sel is None else np.ascontiguousarray(sel, dtype=np.uint8)
    assert sel is None or (alt is not None and alt.shape[1:] == src.shape[1:] and sl.shape == (n,))
    _check(load_library().dmo_gather_rows(context(), src.ptr, None if alt is None else alt.ptr, _ptr(sl), _ptr(idx), n, src.row_elems, out.ptr), "dmo_gather_rows")
    return out


class _Borrowed:
    """Device memory owned by someone else (the mirror of a read-only host array) behind the DeviceArray surface."""

    def __init__(self, ptr, host):
        self.ptr, self.host = ptr, host

    def download(self, count=None):
        return np.array(self.host, dtype=np.float64).reshape(-1)[: None if count is None else int(count)]


def rows_of(a):
    """ResidentRows over ``a``: itself, the device mirror the library already holds for a read-only host array (no
    copy; valid while the mirror lives), or an upload."""
    if isinstance(a, ResidentRows):
        return a
    if isinstance(a, np.ndarray) and a.dtype == np.float64:
        m = mirror_ptr(a)
        if m is not None:
            return ResidentRows(_Borrowed(m, a), a.shape)
    return resident_rows(a)


def scale_rows(rows, factors, seg_row=None, seg_start=None):
    """In place on a ResidentRows: ``rows[seg_row[s]] *= factors[e]`` for e in [seg_start[s], seg_start[s+1]), one rounded
    multiplication after the other (dmo_scale_rows); without segments: ``rows[s] *= factors[s]``."""
    f = _f64(factors)
    sr = None if seg_row is None else np.ascontiguousarray(seg_row, dtype=np.int64)
    ss = None if seg_start is None else np.ascontiguousarray(seg_start, dtype=np.int64)
    n_seg = rows.shape[0] if sr is None else sr.shape[0]
    assert (ss is None or ss.shape[0] == n_seg + 1) and (ss is not None or f.shape[0] == n_seg)
    _check(load_library().dmo_scale_rows(context(), rows.ptr, rows.row_elems, n_seg, _ptr(sr), _ptr(ss), _ptr(f), f.shape[0]), "dmo_scale_rows")
    return rows


def identity_rows(n, d):
    """n copies of the d x d identity, resident (CMAES.py:137-141) -- built on the device from one uploaded matrix."""
    return gather_rows(resident_rows(np.identity(d)[None, :, :]), np.zeros(n, dtype=np.int64))


# --------------------------------------------------------------------------- A13 / A15 CMAES
def cmaes_sample(parents_x, sigmas, A, p_idx, z):
    px = _f64(parents_x)
    sg = _f64(sigmas)
    A = A if isinstance(A, ResidentRows) else _f64(A)
    z = _f64(z)
    pi = np.ascontiguousarray(p_idx, dtype=np.int64)
    n, d = z.shape
    cols = 1 if sg.ndim == 1 else sg.shape[1]
    out = np.empty((n, d), dtype=np.float64)
    _check(load_library().dmo_cmaes_sample(context(), _ptr(px), _ptr(sg), cols, A.ptr if isinstance(A, ResidentRows) else _ptr(A), px.shape[0], _ptr(pi), _ptr(z), n, d,
                                           _ptr(out)), "dmo_cmaes_sample")
    return out


def cmaes_generate(parents_x, sigmas, A, p_idx, z, xlb, xub):
    """Offspring of one MO-CMA-ES generation from the resident parent state: sample, global rescale, clip (CMAES.py:265-270,
    MOEA.py:155) in one call; returns a read-only page-locked (n, d) array whose device copy the next calls reuse."""
    z = _f64(z)
    pi = np.ascontiguousarray(p_idx, dtype=np.int64)
    n, d = z.shape
    px, sg = rows_of(parents_x), rows_of(sigmas)
    cols = 1 if sg.ndim == 1 else sg.shape[1]
    lb, ub = _f64(xlb), _f64(xub)
    x_dev = DeviceArray((n, d), np.float64)
    _check(load_library().dmo_cmaes_generate(context(), px.ptr, sg.ptr, cols, A.ptr, px.shape[0], _ptr(pi), _ptr(z), n, d, _ptr(lb), _ptr(ub), x_dev.ptr),
           "dmo_cmaes_generate")
    out = pinned_empty((n, d), np.float64)
    memcpy(out, x_dev.ptr, out.nbytes)
    mirror_register(out, x_dev)
    out.flags.writeable = False
    return out


def cmaes_step_z(x_gen, cand_idx, parents_x, par_idx, xlb, xub, steps):
    """z = ((x_gen[cand_idx] - parents_x[par_idx]) / (xub - xlb)) / steps on resident rows (CMAES.py:359)."""
    ci = np.ascontiguousarray(cand_idx, dtype=np.int64)
    pi = np.ascontiguousarray(par_idx, dtype=np.int64)
    n, d = ci.shape[0], parents_x.shape[1]
    out = ResidentRows(DeviceArray((n, d), np.float64), (n, d))
    if n:
        lb, ub = _f64(xlb), _f64(xub)
        _check(load_library().dmo_cmaes_step_z(context(), x_gen.ptr, _ptr(ci), parents_x.ptr, _ptr(pi), _ptr(lb), _ptr(ub), steps.ptr, n, d, out.ptr), "dmo_cmaes_step_z")
    return out


def cmaes_update_cholesky(A, Ainv, pc, z, psucc, cc, ccov, pthresh):
    """Batched CMAES.updateCholesky (dmosopt/CMAES.py:489-537); returns new (A, Ainv, pc).  ResidentRows are updated in
    place in HBM (no factor crosses the PCIe bus), host arrays are copied, staged and returned."""
    if isinstance(A, ResidentRows):
        n, d = pc.shape
        if n:
            z, ps = (z if isinstance(z, ResidentRows) else _f64(z)), _f64(psucc)
            _check(load_library().dmo_cmaes_update_cholesky(context(), A.ptr, Ainv.ptr, pc.ptr, _ptr(z), _ptr(ps), n, d, float(cc), float(ccov), float(pthresh)),
                   "dmo_cmaes_update_cholesky")
        return A, Ainv, pc
    A = np.array(A, dtype=np.float64, order="C")
    Ainv = np.array(Ainv, dtype=np.float64, order="C")
    pc = np.array(pc, dtype=np.float64, order="C")
    z = _f64(z)
    ps = _f64(psucc)
    n, d = pc.shape
    _check(load_library().dmo_cmaes_update_cholesky(context(), _ptr(A), _ptr(Ainv), _ptr(pc), _ptr(z), _ptr(ps), n, d, float(cc), float(ccov), float(pthresh)),
           "dmo_cmaes_update_cholesky")
    return A, Ainv, pc
