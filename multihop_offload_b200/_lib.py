"""ctypes binding of libmho.so (include/mho.h).  Fails loudly when the library is missing."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
MAX_F, MAX_K, MAX_LAYERS, MAX_TILE_ROWS = 32, 16, 16, 512
ENV_MAX_NODES, ENV_MAX_LINKS, ENV_MAX_JOBS = 512, 1024, 512
ENV_GREEDY, ENV_LOCAL = 0, 1
ENV_OK, ENV_ROUTE_LOOP, ENV_NO_LINK, ENV_BAD_ITEM = 0, 1, 2, 3


class MhoError(RuntimeError):
    pass


class mho_batch_t(C.Structure):
    _fields_ = [
        ("n_graphs", C.c_int32), ("total_nodes", C.c_int32), ("total_nnz", C.c_int64),
        ("graph_off", C.c_void_p), ("rowptr", C.c_void_p), ("colidx", C.c_void_p), ("vals", C.c_void_p),
        ("rowptr_t", C.c_void_p), ("colidx_t", C.c_void_p), ("vals_t", C.c_void_p),
        ("tile_off", C.c_void_p), ("tile_info", C.c_void_p), ("n_tiles", C.c_int32), ("max_tile_rows", C.c_int32),
        ("max_tile_nnz", C.c_int32), ("adj_bits", C.c_void_p), ("tile_graph0", C.c_void_p),
    ]


class mho_layer_t(C.Structure):
    _fields_ = [("K", C.c_int32), ("f_in", C.c_int32), ("f_out", C.c_int32), ("act", C.c_int32),
                ("slope", C.c_float), ("W", C.c_void_p), ("b", C.c_void_p)]


class mho_head_t(C.Structure):
    _fields_ = [("n_graphs", C.c_int32), ("max_links", C.c_int32), ("total_links", C.c_int64), ("total_comp", C.c_int64),
                ("total_adj_nnz", C.c_int64), ("ext_off", C.c_void_p), ("link_off", C.c_void_p), ("comp_off", C.c_void_p),
                ("maps_ol_el", C.c_void_p), ("maps_on_el", C.c_void_p), ("link_rates", C.c_void_p), ("cf_degs", C.c_void_p),
                ("node_mu", C.c_void_p), ("adj_rowptr", C.c_void_p), ("adj_colidx", C.c_void_p), ("T", C.c_double)]


class mho_env_t(C.Structure):
    _fields_ = [("n_nets", C.c_int32), ("max_nodes", C.c_int32), ("max_links", C.c_int32),
                ("node_off", C.c_void_p), ("link_off", C.c_void_p), ("server_off", C.c_void_p), ("servers", C.c_void_p),
                ("adj_rowptr", C.c_void_p), ("adj_col", C.c_void_p), ("adj_link", C.c_void_p),
                ("link_rates", C.c_void_p), ("cf_degs", C.c_void_p), ("proc_bws", C.c_void_p),
                ("cf_rowptr", C.c_void_p), ("cf_col", C.c_void_p), ("hop", C.c_void_p), ("hop_off", C.c_void_p),
                ("T", C.c_void_p)]


class mho_env_items_t(C.Structure):
    _fields_ = [("n_items", C.c_int32), ("max_jobs", C.c_int32), ("net", C.c_void_p), ("mode", C.c_void_p),
                ("job_off", C.c_void_p), ("sp", C.c_void_p), ("sp_off", C.c_void_p), ("src", C.c_void_p),
                ("rate", C.c_void_p), ("ul", C.c_void_p), ("dl", C.c_void_p)]


class mho_env_out_t(C.Structure):
    _fields_ = [("dst", C.c_void_p), ("nhop", C.c_void_p), ("delay_est", C.c_void_p), ("delay_emp", C.c_void_p),
                ("routes", C.c_void_p), ("routes_off", C.c_void_p), ("route_stride", C.c_int32),
                ("delay_links", C.c_void_p), ("links_off", C.c_void_p), ("delay_nodes", C.c_void_p),
                ("nodes_off", C.c_void_p), ("unit", C.c_void_p), ("unit_off", C.c_void_p), ("status", C.c_void_p)]


class mho_adam_t(C.Structure):
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("clipnorm", C.c_double), ("max_norm", C.c_double), ("decay_rate", C.c_double),
                ("decay_steps", C.c_int32)]


# every symbol include/mho.h declares: (name, restype, argtypes)
PROTOTYPES = [
    ("mho_create", C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    ("mho_destroy", C.c_int, [C.c_void_p]),
    ("mho_last_error", C.c_char_p, []),
    ("mho_version", C.c_int, []),
    ("mho_launch_count", C.c_int64, [C.c_void_p]),
    ("mho_invalidate_weights", C.c_int, [C.c_void_p]),
    ("mho_plan_tiles", C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                 C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("mho_fill_tile_info", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    ("mho_fill_adj_bits", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    ("mho_cheb_forward", C.c_int, [C.c_void_p, C.POINTER(mho_batch_t), C.POINTER(mho_layer_t), C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("mho_saved_bytes", C.c_size_t, [C.POINTER(mho_batch_t), C.POINTER(mho_layer_t), C.c_int32]),
    ("mho_cheb_backward", C.c_int, [C.c_void_p, C.POINTER(mho_batch_t), C.POINTER(mho_layer_t), C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    ("mho_param_count", C.c_int64, [C.POINTER(mho_layer_t), C.c_int32]),
    ("mho_adam_replay", C.c_int, [C.c_void_p, C.POINTER(mho_layer_t), C.c_int32, C.POINTER(mho_adam_t),
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                  C.c_int64, C.c_void_p]),
    ("mho_queue_head_forward", C.c_int, [C.c_void_p, C.POINTER(mho_head_t), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p]),
    ("mho_queue_head_backward", C.c_int, [C.c_void_p, C.POINTER(mho_head_t), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    ("mho_cheb_forward_host_async", C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.POINTER(mho_layer_t), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.POINTER(C.c_int32)]),
    ("mho_host_wait", C.c_int, [C.c_void_p, C.c_int32]),
    ("mho_apsp", C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                           C.c_void_p]),
    ("mho_env_step", C.c_int, [C.c_void_p, C.POINTER(mho_env_t), C.POINTER(mho_env_items_t), C.POINTER(mho_env_out_t),
                               C.c_void_p]),
    ("mho_host_alloc", C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    ("mho_host_free", C.c_int, [C.c_void_p]),
    ("mho_cheb_forward_host", C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(mho_layer_t), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
]


def lib_path():
    return os.environ.get("MHO_LIB", os.path.join(HERE, "libmho.so"))


def load_library():
    """dlopen libmho.so and type every entry point.  No fallback: a missing library is an error."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise MhoError("libmho.so not found at %s - build it with `python -m multihop_offload_b200.build` "
                       "(or __graft_entry__.build()); there is no CPU fallback" % path)
    lib = C.CDLL(path)
    for name, res, args in PROTOTYPES:
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load_library().mho_last_error()
        raise MhoError("%s failed (%d): %s" % (what or "libmho call", rc, (msg or b"").decode()))


class Context:
    """One mho_ctx_t per (process, GPU)."""
    _cache = {}

    def __init__(self, device=0):
        self.lib = load_library()
        self.handle = C.c_void_p()
        check(self.lib.mho_create(C.byref(self.handle), int(device)), "mho_create")
        self.device = int(device)

    @classmethod
    def get(cls, device=0):
        device = int(device)
        if device not in cls._cache:
            cls._cache[device] = cls(device)
        return cls._cache[device]

    def launch_count(self):
        return int(self.lib.mho_launch_count(self.handle))

    def __del__(self):
        try:
            if self.handle:
                self.lib.mho_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass


class PinnedArray:
    """numpy array over a cudaHostAlloc'd buffer (mho_host_alloc); freed with the object."""

    def __init__(self, shape, dtype):
        import numpy as np
        self.lib = load_library()
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        self.ptr = C.c_void_p()
        check(self.lib.mho_host_alloc(C.byref(self.ptr), n), "mho_host_alloc")
        buf = (C.c_char * max(n, 1)).from_address(self.ptr.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            if self.ptr:
                self.array = None
                self.lib.mho_host_free(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


def pinned_like(a):
    """Copy a numpy array into page-locked memory; returns the PinnedArray (use .array)."""
    import numpy as np
    a = np.ascontiguousarray(a)
    p = PinnedArray(a.shape, a.dtype)
    p.array[...] = a
    return p
