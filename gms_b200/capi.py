"""ctypes binding of libgmsb.so (include/gmsb.h).

This is plumbing for tests, bench.py and Python users; the product is the CUDA library.  There is no fallback:
if the shared library is missing or no CUDA device is usable, calls raise.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libgmsb.so")

TC_VARIANTS = {"auto": 0, "merge": 1, "gallop": 2, "bitmap": 3}
EDGE_PASSES = {"auto": 0, "rows": 2, "slots": 3}         # gmsb_tc_options.reserved[3]
SIM_METRICS = {"jaccard": 0, "overlap": 1, "adamic_adar": 2, "resource": 3, "comm_neigh": 4, "total_neigh": 5,
               "pref_att": 6}

_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")


class GmsbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"gmsb error {code}: {msg}")
        self.code = code


class TcOptions(C.Structure):
    _fields_ = [("variant", C.c_int32), ("part_index", C.c_int32), ("part_count", C.c_int32),
                ("reuse_plan", C.c_int32), ("hub_bitmap_bits", C.c_int32), ("gallop_ratio", C.c_int32),
                ("hub_min_work", C.c_int64), ("reserved", C.c_int32 * 4)]


class TcStats(C.Structure):
    _fields_ = [("triangles", C.c_uint64), ("algorithmic_bytes", C.c_uint64), ("wedges_checked", C.c_uint64),
                ("oriented_edges", C.c_int64), ("edges_bitmap", C.c_int64), ("edges_merge", C.c_int64),
                ("edges_gallop", C.c_int64), ("ms_orient", C.c_double), ("ms_count", C.c_double),
                ("ms_bitmap", C.c_double), ("ms_merge", C.c_double), ("ms_gallop", C.c_double),
                ("launches", C.c_int32), ("max_dplus", C.c_int32), ("bytes_bitmap", C.c_uint64),
                ("bytes_light", C.c_uint64), ("wedges_bitmap", C.c_uint64), ("bitmap_items", C.c_int64),
                ("bitmap_smem_bytes", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


# every symbol include/gmsb.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "gmsb_last_error": (C.c_char_p, []),
    "gmsb_version": (C.c_int, []),
    "gmsb_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "gmsb_set_device": (C.c_int, [C.c_int]),
    "gmsb_set_stream": (C.c_int, [C.c_void_p]),
    "gmsb_set_devices": (C.c_int, [C.c_int, C.POINTER(C.c_int)]),
    "gmsb_tc_total_multi": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "gmsb_tc_vertex2_multi": (C.c_int, [C.c_void_p, _i64p]),
    "gmsb_kclique_count_multi": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
    "gmsb_edge_similarity_multi": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int64)]),
    "gmsb_synchronize": (C.c_int, []),
    "gmsb_trim_memory": (C.c_int, []),
    "gmsb_launch_count": (C.c_int, [C.POINTER(C.c_uint64)]),
    "gmsb_generate_rmat": (C.c_int, [C.c_int, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_int, _i32p, _i32p]),
    "gmsb_generate_uniform": (C.c_int, [C.c_int, C.c_int64, _i32p, _i32p]),
    "gmsb_graph_from_csr": (C.c_int, [C.c_int64, _i64p, _i32p, C.c_int, C.POINTER(C.c_void_p)]),
    "gmsb_graph_from_csr_ex": (C.c_int, [C.c_int64, _i64p, _i32p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "gmsb_graph_from_csr_device": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "gmsb_shard_begin": (C.c_int, [C.c_int64, _i64p, _i32p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_int64)]),
    "gmsb_shard_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gmsb_shard_finish": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_void_p)]),
    "gmsb_shard_free": (C.c_int, [C.c_void_p]),
    "gmsb_graph_from_edgelist": (C.c_int, [C.c_int64, _i32p, _i32p, C.c_int, C.POINTER(C.c_void_p)]),
    "gmsb_graph_from_edgelist_device": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_int,
                                                  C.POINTER(C.c_void_p)]),
    "gmsb_graph_relabel_by_degree": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "gmsb_graph_num_nodes": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "gmsb_graph_num_slots": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "gmsb_graph_is_directed": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "gmsb_graph_export_csr": (C.c_int, [C.c_void_p, _i64p, _i32p]),
    "gmsb_graph_free": (C.c_int, [C.c_void_p]),
    "gmsb_order_degree": (C.c_int, [C.c_void_p, C.c_int, _i32p]),
    "gmsb_order_degeneracy": (C.c_int, [C.c_void_p, _i32p]),
    "gmsb_core_numbers": (C.c_int, [C.c_void_p, _i32p]),
    "gmsb_truss_numbers": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "gmsb_order_degeneracy_approx": (C.c_int, [C.c_void_p, C.c_double, C.c_int, _i32p]),
    "gmsb_order_degeneracy_approx_ex": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_int, C.c_uint64, _i32p]),
    "gmsb_graph_worth_relabelling": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "gmsb_orient": (C.c_int, [C.c_void_p, _i32p, C.POINTER(C.c_void_p)]),
    "gmsb_tc_total": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "gmsb_tc_total_ex": (C.c_int, [C.c_void_p, C.POINTER(TcOptions), C.POINTER(C.c_uint64), C.POINTER(TcStats)]),
    "gmsb_tc_vertex2": (C.c_int, [C.c_void_p, _i64p]),
    "gmsb_intersect_count_batch": (C.c_int, [C.c_void_p, C.c_int64, _i32p, _i32p, _u64p]),
    "gmsb_intersect_batch": (C.c_int, [C.c_void_p, C.c_int64, _i32p, _i32p, _i64p, C.c_void_p, C.c_int64]),
    "gmsb_difference_batch": (C.c_int, [C.c_void_p, C.c_int64, _i32p, _i32p, _i64p, C.c_void_p, C.c_int64]),
    "gmsb_union_batch": (C.c_int, [C.c_void_p, C.c_int64, _i32p, _i32p, _i64p, C.c_void_p, C.c_int64]),
    "gmsb_union_count_batch": (C.c_int, [C.c_void_p, C.c_int64, _i32p, _i32p, _u64p]),
    "gmsb_set_from_host": (C.c_int, [_i32p, C.c_int64, C.POINTER(C.c_void_p)]),
    "gmsb_set_range": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p)]),
    "gmsb_set_neighbourhood": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "gmsb_set_clone": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "gmsb_set_free": (C.c_int, [C.c_void_p]),
    "gmsb_set_cardinality": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "gmsb_set_to_host": (C.c_int, [C.c_void_p, _i32p]),
    "gmsb_set_contains": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_int)]),
    "gmsb_set_add": (C.c_int, [C.c_void_p, C.c_int32]),
    "gmsb_set_remove": (C.c_int, [C.c_void_p, C.c_int32]),
    "gmsb_set_equal": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "gmsb_set_op": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "gmsb_set_op_inplace": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "gmsb_set_op_count": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    "gmsb_set_op_count_many": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p), _u64p]),
    "gmsb_set_op_many": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "gmsb_set_op_count_neighbourhoods": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, _u64p]),
    "gmsb_pair_similarity": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, _i32p, _i32p, _f64p]),
    "gmsb_edge_similarity": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int64)]),
    "gmsb_kclique_count": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
    "gmsb_kclique_count_ex": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64)]),
    "gmsb_kclique_count_ordered": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
}

_lib = None


def lib():
    """Load libgmsb.so; raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `make -C gms_b200/csrc` "
                              "(gms-b200 has no CPU fallback)")
        dll = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(dll, name)
            f.restype, f.argtypes = res, args
        _lib = dll
    return _lib


def _check(code):
    if code != 0:
        raise GmsbError(code, lib().gmsb_last_error().decode())


def device_count():
    c = C.c_int(0)
    _check(lib().gmsb_device_count(C.byref(c)))
    return c.value


def set_device(i):
    _check(lib().gmsb_set_device(i))


def _bundled_nccl():
    """Path of the pip-installed NCCL (the nvidia-nccl wheel PyTorch depends on), or None.  The multi-GPU entry points
    dlopen libnccl.so.2; a process that later imports torch must get the SAME file, because the loader keeps one object
    per SONAME (an older system libnccl opened first would leave torch without the symbols it was built against)."""
    import importlib.util
    try:
        spec = importlib.util.find_spec("nvidia.nccl")
    except (ImportError, ValueError):
        return None
    for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
        path = os.path.join(base, "lib", "libnccl.so.2")
        if os.path.exists(path):
            return path
    return None


def set_devices(ids):
    """The devices of the *_multi entry points (one process, several GPUs); ids[0] becomes the primary device."""
    if len(ids) > 1 and not os.environ.get("GMSB_NCCL_LIB"):
        path = _bundled_nccl()
        if path:
            os.environ["GMSB_NCCL_LIB"] = path          # read by the library when it first reduces an array (mgpu.cu)
    arr = (C.c_int * len(ids))(*ids)
    _check(lib().gmsb_set_devices(len(ids), arr))


def set_stream(ptr):
    _check(lib().gmsb_set_stream(ptr))


def synchronize():
    _check(lib().gmsb_synchronize())


def launch_count():
    c = C.c_uint64(0)
    _check(lib().gmsb_launch_count(C.byref(c)))
    return c.value


def generate_rmat(scale, m=None, a=0.57, b=0.19, c=0.19, permute=True, degree=16):
    """Reference generator semantics (gapbs/generator.h:81-114); defaults = `-g kronecker <scale> --deg 16`."""
    m = (1 << scale) * degree if m is None else m
    src, dst = np.zeros(max(m, 1), np.int32), np.zeros(max(m, 1), np.int32)
    _check(lib().gmsb_generate_rmat(scale, m, a, b, c, int(permute), src, dst))
    return src[:m], dst[:m]


def generate_uniform(scale, m=None, degree=16):
    m = (1 << scale) * degree if m is None else m
    src, dst = np.zeros(max(m, 1), np.int32), np.zeros(max(m, 1), np.int32)
    _check(lib().gmsb_generate_uniform(scale, m, src, dst))
    return src[:m], dst[:m]


def _ids(x):
    x = np.ascontiguousarray(x, np.int32)
    return x if len(x) else np.zeros(1, np.int32)


class Graph:
    """A device-resident CSR graph (the SGraph of the reference's algorithms)."""

    def __init__(self, handle):
        self.h = C.c_void_p(handle) if not isinstance(handle, C.c_void_p) else handle

    # --- construction
    @staticmethod
    def from_csr(offsets, nbrs, directed=False, orient=False):
        """orient=True: GMSB_BUILD_ORIENT — the degree-oriented representation is built while the arrays upload."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        n = len(offsets) - 1
        nn = len(nbrs)
        h = C.c_void_p()
        if orient:
            _check(lib().gmsb_graph_from_csr_ex(n, offsets, _ids(nbrs), int(directed), 1, C.byref(h)))
        else:
            _check(lib().gmsb_graph_from_csr(n, offsets, _ids(nbrs), int(directed), C.byref(h)))
        assert nn >= offsets[-1]
        return Graph(h)

    @staticmethod
    def from_csr_device(n, offsets_ptr, nbrs_ptr, directed=False):
        h = C.c_void_p()
        _check(lib().gmsb_graph_from_csr_device(n, offsets_ptr, nbrs_ptr, int(directed), C.byref(h)))
        return Graph(h)

    @staticmethod
    def from_edgelist(src, dst, symmetrize=True):
        assert len(src) == len(dst)
        h = C.c_void_p()
        _check(lib().gmsb_graph_from_edgelist(len(src), _ids(src), _ids(dst), int(symmetrize), C.byref(h)))
        return Graph(h)

    @staticmethod
    def from_edgelist_device(m, src_ptr, dst_ptr, symmetrize=True):
        h = C.c_void_p()
        _check(lib().gmsb_graph_from_edgelist_device(m, src_ptr, dst_ptr, int(symmetrize), C.byref(h)))
        return Graph(h)

    def free(self):
        if self.h:
            lib().gmsb_graph_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    # --- properties
    @property
    def n(self):
        v = C.c_int64(0)
        _check(lib().gmsb_graph_num_nodes(self.h, C.byref(v)))
        return v.value

    @property
    def slots(self):
        v = C.c_int64(0)
        _check(lib().gmsb_graph_num_slots(self.h, C.byref(v)))
        return v.value

    @property
    def directed(self):
        v = C.c_int(0)
        _check(lib().gmsb_graph_is_directed(self.h, C.byref(v)))
        return bool(v.value)

    def export_csr(self):
        off = np.zeros(self.n + 1, np.int64)
        nbr = np.zeros(max(self.slots, 1), np.int32)
        _check(lib().gmsb_graph_export_csr(self.h, off, nbr))
        return off, nbr[:off[-1]]

    # --- transforms / orderings
    def relabel_by_degree(self):
        h = C.c_void_p()
        _check(lib().gmsb_graph_relabel_by_degree(self.h, C.byref(h)))
        return Graph(h)

    def degree_order(self, rank_format=False):
        out = np.zeros(max(self.n, 1), np.int32)
        _check(lib().gmsb_order_degree(self.h, int(rank_format), out))
        return out[:self.n]

    def degeneracy_rank(self):
        out = np.zeros(max(self.n, 1), np.int32)
        _check(lib().gmsb_order_degeneracy(self.h, out))
        return out[:self.n]

    def core_numbers(self):
        """Core number of every vertex (int32[n]); the maximum is the degeneracy."""
        out = np.zeros(max(self.n, 1), np.int32)
        _check(lib().gmsb_core_numbers(self.h, out))
        return out[:self.n]

    def truss_numbers(self):
        """Truss number of every undirected edge u<v (int32[m]), in the edge order of edge_similarity."""
        m = C.c_int64(0)
        _check(lib().gmsb_truss_numbers(self.h, None, C.byref(m)))
        out = np.zeros(max(m.value, 1), np.int32)
        _check(lib().gmsb_truss_numbers(self.h, out.ctypes.data, C.byref(m)))
        return out[:m.value]

    def degeneracy_order_approx(self, epsilon=1.0, rank_format=False):
        out = np.zeros(max(self.n, 1), np.int32)
        _check(lib().gmsb_order_degeneracy_approx(self.h, float(epsilon), int(rank_format), out))
        return out[:self.n]

    def degeneracy_order_approx_ex(self, epsilon=1.0, rank_format=False, boundary="average", pull=False, seed=1):
        kinds = {"average": 0, "min": 1, "prob_min": 2, "prob_median": 3}
        out = np.zeros(max(self.n, 1), np.int32)
        _check(lib().gmsb_order_degeneracy_approx_ex(self.h, float(epsilon), int(rank_format), kinds[boundary], int(pull),
                                                     seed, out))
        return out[:self.n]

    def worth_relabelling(self):
        v = C.c_int(0)
        _check(lib().gmsb_graph_worth_relabelling(self.h, C.byref(v)))
        return bool(v.value)

    def orient(self, ranking):
        h = C.c_void_p()
        _check(lib().gmsb_orient(self.h, _ids(ranking), C.byref(h)))
        return Graph(h)

    # --- triangles
    def tc_total(self):
        out = C.c_uint64(0)
        _check(lib().gmsb_tc_total(self.h, C.byref(out)))
        return out.value

    def tc_total_ex(self, variant="auto", part_index=0, part_count=1, reuse_plan=False, hub_bitmap_bits=0,
                    gallop_ratio=0, hub_min_work=0, edge_passes="auto"):
        """Triangle count with options (gmsb_tc_options); returns (count, statistics as a dict).

        With part_count > 1 the count and the statistics cover share part_index of the oriented edges.  edge_passes
        picks the form of the schedule's two passes over the edges: "rows" walks the rows, "slots" streams over the
        edge slots, "auto" takes the element-wise form from 4 parts on.  Both forms build the same schedule."""
        opt = TcOptions(TC_VARIANTS[variant], part_index, part_count, int(reuse_plan), hub_bitmap_bits, gallop_ratio,
                        hub_min_work, (C.c_int32 * 4)(0, 0, 0, EDGE_PASSES[edge_passes]))
        out, st = C.c_uint64(0), TcStats()
        _check(lib().gmsb_tc_total_ex(self.h, C.byref(opt), C.byref(out), C.byref(st)))
        return out.value, st.as_dict()

    def tc_vertex2(self):
        out = np.zeros(max(self.n, 1), np.int64)
        _check(lib().gmsb_tc_vertex2(self.h, out))
        return out[:self.n]

    # --- set algebra / similarity
    def intersect_count_batch(self, a, b):
        assert len(a) == len(b)
        out = np.zeros(max(len(a), 1), np.uint64)
        _check(lib().gmsb_intersect_count_batch(self.h, len(a), _ids(a), _ids(b), out))
        return out[:len(a)]

    def _two_pass(self, fn, a, b):
        assert len(a) == len(b)
        off = np.zeros(len(a) + 1, np.int64)
        _check(fn(self.h, len(a), _ids(a), _ids(b), off, None, 0))
        elems = np.zeros(max(int(off[-1]), 1), np.int32)
        _check(fn(self.h, len(a), _ids(a), _ids(b), off, elems.ctypes.data, len(elems)))
        return off, elems[:off[-1]]

    def intersect_batch(self, a, b):
        return self._two_pass(lib().gmsb_intersect_batch, a, b)

    def difference_batch(self, a, b):
        """N(a[i]) \\ N(b[i]) for every pair: (offsets, elements), ascending inside each result."""
        return self._two_pass(lib().gmsb_difference_batch, a, b)

    def union_batch(self, a, b):
        return self._two_pass(lib().gmsb_union_batch, a, b)

    def union_count_batch(self, a, b):
        assert len(a) == len(b)
        out = np.zeros(max(len(a), 1), np.uint64)
        _check(lib().gmsb_union_count_batch(self.h, len(a), _ids(a), _ids(b), out))
        return out[:len(a)]

    def pair_similarity(self, metric, a, b):
        assert len(a) == len(b)
        out = np.zeros(max(len(a), 1), np.float64)
        _check(lib().gmsb_pair_similarity(self.h, SIM_METRICS[metric], len(a), _ids(a), _ids(b), out))
        return out[:len(a)]

    def edge_similarity(self, metric):
        m = C.c_int64(0)
        _check(lib().gmsb_edge_similarity(self.h, SIM_METRICS[metric], None, C.byref(m)))
        out = np.zeros(max(m.value, 1), np.float64)
        _check(lib().gmsb_edge_similarity(self.h, SIM_METRICS[metric], out.ctypes.data, C.byref(m)))
        return out[:m.value]

    # --- several GPUs in one process (after gms_b200.set_devices)
    def tc_total_multi(self):
        out = C.c_uint64(0)
        _check(lib().gmsb_tc_total_multi(self.h, C.byref(out)))
        return out.value

    def tc_vertex2_multi(self):
        out = np.zeros(max(self.n, 1), np.int64)
        _check(lib().gmsb_tc_vertex2_multi(self.h, out))
        return out[:self.n]

    def kclique_count_multi(self, k):
        out = C.c_uint64(0)
        _check(lib().gmsb_kclique_count_multi(self.h, k, C.byref(out)))
        return out.value

    def edge_similarity_multi(self, metric):
        m = C.c_int64(0)
        _check(lib().gmsb_edge_similarity_multi(self.h, SIM_METRICS[metric], None, C.byref(m)))
        out = np.zeros(max(m.value, 1), np.float64)
        _check(lib().gmsb_edge_similarity_multi(self.h, SIM_METRICS[metric], out.ctypes.data, C.byref(m)))
        return out[:m.value]

    # --- cliques
    def kclique_count(self, k, part_index=0, part_count=1):
        out = C.c_uint64(0)
        _check(lib().gmsb_kclique_count_ex(self.h, k, part_index, part_count, C.byref(out)))
        return out.value

    def kclique_count_ordered(self, k):
        out = C.c_uint64(0)
        _check(lib().gmsb_kclique_count_ordered(self.h, k, C.byref(out)))
        return out.value


SET_OPS = {"intersect": 0, "union": 1, "difference": 2}


class Shard:
    """One device's share of a sharded build of the oriented representation (gmsb_shard_*): `begin` uploads and orients
    the vertex range of part `part_index`; the caller exchanges the exported pieces; `finish` returns a Graph that
    answers the triangle entry points."""

    def __init__(self, offsets, nbrs, part_index, part_count, offsets_dev_ptr=None):
        """offsets_dev_ptr: device pointer of the complete int64 offsets (e.g. after an all-gather), or None to upload
        them from `offsets`."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        h, plen = C.c_void_p(), C.c_int64()
        _check(lib().gmsb_shard_begin(len(offsets) - 1, offsets, _ids(nbrs),
                                      C.c_void_p(offsets_dev_ptr) if offsets_dev_ptr else None, int(part_index),
                                      int(part_count), C.byref(h), C.byref(plen)))
        self.h, self.piece_len = h, plen.value

    def export(self, piece_ptr, dplus_all_ptr):
        """piece_ptr: device int32[>= piece_len]; dplus_all_ptr: device int32[n], zeroed by the caller."""
        _check(lib().gmsb_shard_export(self.h, C.c_void_p(piece_ptr), C.c_void_p(dplus_all_ptr)))

    def finish(self, pieces_ptr, piece_stride, dplus_all_ptr):
        g = C.c_void_p()
        _check(lib().gmsb_shard_finish(self.h, C.c_void_p(pieces_ptr), int(piece_stride), C.c_void_p(dplus_all_ptr),
                                       C.byref(g)))
        self.free()
        return Graph(g)

    def free(self):
        if self.h:
            lib().gmsb_shard_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DeviceSet:
    """Device-resident sorted set (gmsb_set_*): the reference's Set concept (sorted_set.h) with results kept in HBM."""

    def __init__(self, elems=(), _h=None):
        if _h is not None:
            self.h = _h
            return
        h = C.c_void_p()
        arr = np.ascontiguousarray(elems, np.int32)
        _check(lib().gmsb_set_from_host(_ids(arr), len(arr), C.byref(h)))
        self.h = h

    def __del__(self):
        if getattr(self, "h", None):
            lib().gmsb_set_free(self.h)
            self.h = None

    @staticmethod
    def range(bound):
        h = C.c_void_p()
        _check(lib().gmsb_set_range(bound, C.byref(h)))
        return DeviceSet(_h=h)

    @staticmethod
    def neighbourhood(graph, v):
        h = C.c_void_p()
        _check(lib().gmsb_set_neighbourhood(graph.h, v, C.byref(h)))
        s = DeviceSet(_h=h)
        s._graph = graph                      # the view borrows the graph's CSR
        return s

    def clone(self):
        h = C.c_void_p()
        _check(lib().gmsb_set_clone(self.h, C.byref(h)))
        return DeviceSet(_h=h)

    def cardinality(self):
        n = C.c_int64(0)
        _check(lib().gmsb_set_cardinality(self.h, C.byref(n)))
        return n.value

    def to_array(self):
        out = np.zeros(max(self.cardinality(), 1), np.int32)
        _check(lib().gmsb_set_to_host(self.h, out))
        return out[:self.cardinality()]

    def contains(self, x):
        f = C.c_int(0)
        _check(lib().gmsb_set_contains(self.h, x, C.byref(f)))
        return bool(f.value)

    def add(self, x):
        _check(lib().gmsb_set_add(self.h, x))

    def remove(self, x):
        _check(lib().gmsb_set_remove(self.h, x))

    def __eq__(self, other):
        f = C.c_int(0)
        _check(lib().gmsb_set_equal(self.h, other.h, C.byref(f)))
        return bool(f.value)

    def op(self, kind, other):
        h = C.c_void_p()
        _check(lib().gmsb_set_op(SET_OPS[kind], self.h, other.h, C.byref(h)))
        return DeviceSet(_h=h)

    def op_inplace(self, kind, other):
        _check(lib().gmsb_set_op_inplace(SET_OPS[kind], self.h, other.h))

    def op_count(self, kind, other):
        out = C.c_uint64(0)
        _check(lib().gmsb_set_op_count(SET_OPS[kind], self.h, other.h, C.byref(out)))
        return out.value

    def op_count_many(self, kind, others):
        hs = (C.c_void_p * max(len(others), 1))(*[o.h for o in others])
        out = np.zeros(max(len(others), 1), np.uint64)
        _check(lib().gmsb_set_op_count_many(SET_OPS[kind], self.h, len(others), hs, out))
        return out[:len(others)]

    def op_many(self, kind, others):
        hs = (C.c_void_p * max(len(others), 1))(*[o.h for o in others])
        outs = (C.c_void_p * max(len(others), 1))()
        _check(lib().gmsb_set_op_many(SET_OPS[kind], self.h, len(others), hs, outs))
        return [DeviceSet(_h=C.c_void_p(outs[i])) for i in range(len(others))]

    def op_count_neighbourhoods(self, kind, graph, members):
        out = np.zeros(max(members.cardinality(), 1), np.uint64)
        _check(lib().gmsb_set_op_count_neighbourhoods(SET_OPS[kind], self.h, graph.h, members.h, out))
        return out[:members.cardinality()]
