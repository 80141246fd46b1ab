"""ctypes binding of the C ABI in include/graph_embed_b200.h.

This is what tests/ and bench.py call: numpy/scipy host buffers in, numpy out, every call going
through the same `extern "C"` entry points a C++ / cgo / JNI caller would bind.  There is no
Python or CPU implementation behind these functions: if the shared library is missing the import
of the library fails loudly, and every compute entry point returns GE_ERR_NO_DEVICE without a B200.
"""
import ctypes as C
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
# GE_LIB: an alternative build of the same library (kernel experiments: tools/sweep_*.py)
LIB_PATH = os.environ.get("GE_LIB") or os.path.join(PKG, "lib", "libgraphembed_b200.so")

GE_OK, GE_ERR_INVALID, GE_ERR_NO_DEVICE, GE_ERR_CUDA, GE_ERR_OOM, GE_ERR_UNSUPPORTED = range(6)
GE_F64, GE_F32 = 0, 1

_pi = C.POINTER(C.c_int32)
_pd = C.POINTER(C.c_double)


class GeError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("graph_embed_b200 status %d: %s" % (status, message))
        self.status = status


class Csr(C.Structure):
    _fields_ = [("rows", C.c_int32), ("cols", C.c_int32), ("nnz", C.c_int64),
                ("indptr", _pi), ("indices", _pi), ("data", _pd)]


class Params(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("ks", C.c_double), ("ksmax", C.c_double),
                ("repel", C.c_double), ("attract", C.c_double), ("gravity", C.c_double),
                ("delta", C.c_double), ("tolerate", C.c_double), ("use_weights", C.c_int32),
                ("linlog", C.c_int32), ("nohubs", C.c_int32), ("normalize", C.c_int32),
                ("precision", C.c_int32), ("seed", C.c_uint32)]


class EmbedOptions(C.Structure):
    _fields_ = [("coarse_iterations", C.c_int32), ("level_iterations", C.c_int32),
                ("precision", C.c_int32), ("seed", C.c_uint32), ("verbose", C.c_int32),
                ("first_layer", C.c_int32)]


class EmbedStats(C.Structure):
    _fields_ = [("total_ms", C.c_double), ("coarse_ms", C.c_double), ("levels_ms", C.c_double),
                ("host_radii_ms", C.c_double), ("h2d_bytes", C.c_double), ("d2h_bytes", C.c_double),
                ("pair_interactions", C.c_double), ("edge_visits", C.c_double),
                ("kernel_launches", C.c_int64), ("grid_tier_ms", C.c_double),
                ("device_radii_ms", C.c_double)]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


# every symbol include/graph_embed_b200.h declares (tests check the library exports them all)
SYMBOLS = [
    "ge_version", "ge_last_error", "ge_params_default_flat", "ge_params_default_multilevel",
    "ge_embed_options_default", "ge_context_create", "ge_context_destroy",
    "ge_context_launch_count", "ge_context_bytes", "ge_measure_fma_peak",
    "ge_flat_forceatlas", "ge_multilevel_forceatlas", "ge_multilevel_forceatlas_shard", "ge_embed",
    "ge_flat_forces", "ge_multilevel_forces", "ge_level_radii", "ge_reference_uniform",
    "ge_flat_plan_create", "ge_flat_plan_destroy", "ge_flat_plan_ld", "ge_flat_plan_elem_size",
    "ge_flat_plan_bind_coords", "ge_flat_plan_upload_coords", "ge_flat_plan_download_coords",
    "ge_flat_plan_download_forces", "ge_flat_plan_cur_coords", "ge_flat_plan_next_coords",
    "ge_flat_plan_launch_iteration", "ge_flat_plan_swap", "ge_flat_plan_iterate",
    "ge_flat_plan_sync", "ge_flat_plan_select_kernels", "ge_flat_plan_profile", "ge_flat_plan_profile_get",
    "ge_flat_plan_create_symmetric", "ge_flat_plan_is_symmetric", "ge_flat_plan_pair_sums",
    "ge_flat_plan_bind_pair_sums", "ge_flat_plan_launch_repulsion", "ge_flat_plan_launch_step",
    "ge_flat_symmetric_share", "ge_galerkin", "ge_level_radii_device",
    "ge_context_create_multi", "ge_context_device_count",
    "ge_flat_symmetric_pass_share", "ge_embed_aggregate_ranges", "ge_embed_aggregate_owners",
    "ge_coarsen_options_default", "ge_coarsen", "ge_hierarchy_levels", "ge_hierarchy_graph",
    "ge_hierarchy_aggregation", "ge_hierarchy_destroy", "ge_largest_component", "ge_layout_graph",
    "ge_edges_options_default", "ge_graph_from_edges", "ge_layout_edges",
]

_lib = None


def lib():
    """Loads lib/libgraphembed_b200.so; raises if it was not built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: run `python graph-embed_b200/build.py` "
                              "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.ge_version.restype = C.c_char_p
        L.ge_last_error.restype = C.c_char_p
        L.ge_context_launch_count.restype = C.c_int64
        L.ge_flat_plan_ld.restype = C.c_int64
        L.ge_flat_plan_cur_coords.restype = C.c_void_p
        L.ge_flat_plan_next_coords.restype = C.c_void_p
        L.ge_flat_plan_pair_sums.restype = C.c_void_p
        L.ge_flat_plan_is_symmetric.restype = C.c_int32
        L.ge_reference_uniform.argtypes = [C.c_uint32, C.c_int64, _pd]
        L.ge_context_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
        L.ge_context_bytes.restype = None
        L.ge_hierarchy_levels.argtypes = [C.c_void_p]
        L.ge_hierarchy_levels.restype = C.c_int32
        for name in ("ge_context_destroy", "ge_flat_plan_destroy", "ge_flat_plan_swap", "ge_hierarchy_destroy"):
            getattr(L, name).argtypes = [C.c_void_p]
            getattr(L, name).restype = None
        _lib = L
    return _lib


def _check(status):
    if status != GE_OK:
        raise GeError(status, lib().ge_last_error().decode())


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a, typ):
    return None if a is None else a.ctypes.data_as(typ)


class GalerkinStats(C.Structure):
    _fields_ = [("device_ms", C.c_double), ("total_ms", C.c_double), ("kernel_launches", C.c_int64),
                ("segments_shared", C.c_int64), ("segments_global", C.c_int64), ("nnz_out", C.c_int64)]


class CoarsenOptions(C.Structure):
    _fields_ = [("coarsening_factor", C.c_double), ("min_coarse", C.c_int32), ("max_levels", C.c_int32),
                ("seed", C.c_uint32)]


class CoarsenStats(C.Structure):
    _fields_ = [("total_ms", C.c_double), ("device_ms", C.c_double), ("rounds", C.c_int64),
                ("kernel_launches", C.c_int64)]


class LayoutStats(C.Structure):
    _fields_ = [("total_ms", C.c_double), ("components_ms", C.c_double), ("coarsen_ms", C.c_double),
                ("embed_ms", C.c_double), ("components", C.c_int64), ("levels", C.c_int32),
                ("h2d_bytes", C.c_double), ("d2h_bytes", C.c_double), ("kernel_launches", C.c_int64)]


class EdgesOptions(C.Structure):
    _fields_ = [("symmetrize", C.c_int32), ("keep_self_loops", C.c_int32), ("unit_weights", C.c_int32)]


class EdgesStats(C.Structure):
    _fields_ = [("total_ms", C.c_double), ("device_ms", C.c_double), ("nnz", C.c_int64),
                ("self_loops_dropped", C.c_int64), ("duplicates_merged", C.c_int64),
                ("kernel_launches", C.c_int64)]


def _struct_dict(st):
    return {f: getattr(st, f) for f, _ in st._fields_}


class EdgeList:
    """int32 id arrays (and float64 weights) of an edge list, checked to fit the C ABI's int32 ids."""

    def __init__(self, n, src, dst, weights=None):
        src, dst = np.asarray(src).ravel(), np.asarray(dst).ravel()
        if src.shape != dst.shape:
            raise ValueError("src and dst differ in length")
        if src.size and not (np.issubdtype(src.dtype, np.integer) and np.issubdtype(dst.dtype, np.integer)):
            raise ValueError("vertex ids must be integers")
        lo, hi = np.iinfo(np.int32).min, np.iinfo(np.int32).max
        if not lo <= int(n) <= hi:
            raise GeError(GE_ERR_INVALID, "n does not fit int32")
        for a in (src, dst):  # ids of a wider type must fit int32 before they are narrowed
            if a.size and a.dtype != np.int32 and (int(a.min()) < lo or int(a.max()) > hi):
                raise GeError(GE_ERR_INVALID, "a vertex id does not fit int32")
        self.n, self.E = int(n), int(src.size)
        self.src, self.dst = _i32(src), _i32(dst)
        self.w = None if weights is None else _f64(np.asarray(weights).ravel())
        if self.w is not None and self.w.size != self.E:
            raise ValueError("weights differ in length from the edges")

    def args(self):
        return (C.c_int32(self.n), C.c_int64(self.E), _ptr(self.src, _pi), _ptr(self.dst, _pi), _ptr(self.w, _pd))


def edges_options(symmetrize=True, keep_self_loops=False, unit_weights=False):
    o = EdgesOptions()
    lib().ge_edges_options_default(C.byref(o))
    o.symmetrize, o.keep_self_loops, o.unit_weights = int(bool(symmetrize)), int(bool(keep_self_loops)), \
        int(bool(unit_weights))
    return o


def _csr_copy(c, with_data=True):
    """scipy CSR copy of a ge_csr view (int32 / float64)."""
    import scipy.sparse as sp
    nnz = int(c.nnz)
    indptr = np.ctypeslib.as_array(c.indptr, shape=(c.rows + 1,)).copy()
    indices = np.ctypeslib.as_array(c.indices, shape=(nnz,)).copy() if nnz else np.zeros(0, np.int32)
    data = np.ctypeslib.as_array(c.data, shape=(nnz,)).copy() if nnz else np.zeros(0)
    return sp.csr_matrix((data, indices, indptr), shape=(c.rows, c.cols))


class CsrView:
    """Keeps the numpy arrays of a scipy CSR alive next to the ge_csr that points into them."""

    def __init__(self, A, with_data=True):
        self.indptr, self.indices = _i32(A.indptr), _i32(A.indices)
        self.data = _f64(A.data) if with_data else None
        self.c = Csr(A.shape[0], A.shape[1], int(self.indptr[-1]), _ptr(self.indptr, _pi),
                     _ptr(self.indices, _pi), _ptr(self.data, _pd))

    def ref(self):
        return C.byref(self.c)


def flat_params(**kw):
    p = Params()
    lib().ge_params_default_flat(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def multilevel_params(**kw):
    p = Params()
    lib().ge_params_default_multilevel(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def vertex_to_aggregate(P_T):
    v_A = np.empty(P_T.shape[1], dtype=np.int32)
    v_A[P_T.indices] = np.repeat(np.arange(P_T.shape[0], dtype=np.int32), np.diff(P_T.indptr))
    return v_A


def reference_uniform(seed, count):
    out = np.zeros(int(count))
    lib().ge_reference_uniform(int(seed), int(count), _ptr(out, _pd))
    return out


def level_radii(coords_A, dim, A_c=None, P_T_c=None, coords_Ac=None, r_Ac=None):
    """src/embed.cpp:615-778 through ge_level_radii (host only) -> (coords_A, r_A)."""
    cA = _f64(coords_A).reshape(-1, dim).copy()
    m = cA.shape[0]
    rA = np.zeros(m)
    if P_T_c is None:
        _check(lib().ge_level_radii(m, dim, _ptr(cA, _pd), _ptr(rA, _pd), None, None, None, None))
    else:
        Ac, Pc = CsrView(A_c), CsrView(P_T_c, with_data=False)
        cAc, rAc = _f64(coords_Ac).reshape(-1, dim), _f64(r_Ac)
        _check(lib().ge_level_radii(m, dim, _ptr(cA, _pd), _ptr(rA, _pd), Ac.ref(), Pc.ref(),
                                    _ptr(cAc, _pd), _ptr(rAc, _pd)))
    return cA, rA


class Context:
    """ge_context: one device + stream.  Raises GeError(GE_ERR_NO_DEVICE) without a B200."""

    def __init__(self, device=-1, stream=None, devices=None):
        """devices=[d0, d1, ...]: one context over several GPUs (ge_context_create_multi)."""
        self.h = C.c_void_p()
        if devices is not None:
            ids = (C.c_int * len(devices))(*[int(d) for d in devices])
            _check(lib().ge_context_create_multi(len(devices), ids, C.byref(self.h)))
        else:
            _check(lib().ge_context_create(int(device), C.c_void_p(stream) if stream else None,
                                           C.byref(self.h)))

    @property
    def device_count(self):
        return int(lib().ge_context_device_count(self.h))

    def close(self):
        if self.h:
            lib().ge_context_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return int(lib().ge_context_launch_count(self.h))

    @property
    def bytes_moved(self):
        h2d, d2h = C.c_double(), C.c_double()
        lib().ge_context_bytes(self.h, C.byref(h2d), C.byref(d2h))
        return h2d.value, d2h.value

    def fma_peak_tflops(self, precision=GE_F64):
        t = C.c_double()
        _check(lib().ge_measure_fma_peak(self.h, int(precision), C.byref(t)))
        return t.value

    # -- the reference's kernels, host buffers ------------------------------------------------
    def flat_forceatlas(self, A, dim, coords, params, inplace=False):
        a = CsrView(A)
        x = _f64(coords).reshape(A.shape[0], dim)
        if not inplace:
            x = x.copy()
        _check(lib().ge_flat_forceatlas(self.h, a.ref(), int(dim), _ptr(x, _pd), C.byref(params)))
        return x

    def multilevel_forceatlas(self, A, P_T, coords_A, r_A, dim, params, init=None, aggregates=None):
        """aggregates=(begin, end): solve only that range (rows of other aggregates come back 0)."""
        a, p = CsrView(A), CsrView(P_T, with_data=False)
        n, m = A.shape[0], P_T.shape[0]
        v_A = vertex_to_aggregate(P_T)
        cA, rA = _f64(coords_A).reshape(m, dim), _f64(r_A)
        x0 = None if init is None else _f64(init).reshape(n, dim)
        out = np.zeros((n, dim))
        if aggregates is None:
            _check(lib().ge_multilevel_forceatlas(self.h, a.ref(), p.ref(), _ptr(v_A, _pi),
                                                  _ptr(cA, _pd), _ptr(rA, _pd), _ptr(x0, _pd),
                                                  _ptr(out, _pd), int(dim), C.byref(params)))
        else:
            _check(lib().ge_multilevel_forceatlas_shard(
                self.h, a.ref(), p.ref(), _ptr(v_A, _pi), _ptr(cA, _pd), _ptr(rA, _pd), _ptr(x0, _pd),
                _ptr(out, _pd), int(dim), C.byref(params), int(aggregates[0]), int(aggregates[1])))
        return out

    def embed(self, As, P_Ts, dim, seed=0, precision=GE_F64, coarse_iterations=100000,
              level_iterations=100, verbose=False, return_level1=False):
        L = len(P_Ts)
        assert len(As) == L + 1
        av = [CsrView(A) for A in As]
        pv = [CsrView(P, with_data=False) for P in P_Ts]
        a_arr = (Csr * (L + 1))(*[v.c for v in av])
        p_arr = (Csr * max(L, 1))(*([v.c for v in pv] or [Csr()]))
        opt = EmbedOptions()
        lib().ge_embed_options_default(C.byref(opt))
        opt.seed, opt.precision, opt.verbose = int(seed), int(precision), int(verbose)
        opt.coarse_iterations, opt.level_iterations = int(coarse_iterations), int(level_iterations)
        out = np.zeros((As[0].shape[0], dim))
        m = As[1].shape[0] if L else 0
        r_A, coords_A = np.zeros(max(m, 1)), np.zeros((max(m, 1), dim))
        stats = EmbedStats()
        # embedMultilevel's out-parameters (level 1's radii / rescaled coordinates) are copied back
        # only on request: partition::embed itself returns the finest coordinates alone
        _check(lib().ge_embed(self.h, L, a_arr, p_arr, int(dim), C.byref(opt), _ptr(out, _pd),
                              _ptr(r_A, _pd) if return_level1 else None,
                              _ptr(coords_A, _pd) if return_level1 else None, C.byref(stats)))
        if return_level1:
            return out, stats.as_dict(), r_A[:m], coords_A[:m]
        return out, stats.as_dict()

    def level_radii(self, coords_A, dim, A_c=None, P_T_c=None, coords_Ac=None, r_Ac=None):
        """src/embed.cpp:615-778 on the device (ge_level_radii_device) -> (coords_A, r_A)."""
        cA = _f64(coords_A).reshape(-1, dim).copy()
        m = cA.shape[0]
        rA = np.zeros(m)
        if P_T_c is None:
            _check(lib().ge_level_radii_device(self.h, m, dim, _ptr(cA, _pd), _ptr(rA, _pd), None, None, None, None))
        else:
            Ac, Pc = CsrView(A_c), CsrView(P_T_c, with_data=False)
            cAc, rAc = _f64(coords_Ac).reshape(-1, dim), _f64(r_Ac)
            _check(lib().ge_level_radii_device(self.h, m, dim, _ptr(cA, _pd), _ptr(rA, _pd), Ac.ref(), Pc.ref(),
                                               _ptr(cAc, _pd), _ptr(rAc, _pd)))
        return cA, rA

    # -- parity hooks -------------------------------------------------------------------------
    def flat_forces(self, A, dim, coords, params, path=0):
        a = CsrView(A)
        x = _f64(coords).reshape(A.shape[0], dim)
        F = np.zeros((A.shape[0], dim))
        _check(lib().ge_flat_forces(self.h, a.ref(), int(dim), _ptr(x, _pd), C.byref(params),
                                    int(path), _ptr(F, _pd)))
        return F

    def multilevel_forces(self, A, P_T, coords_A, positions, dim, params):
        a, p = CsrView(A), CsrView(P_T, with_data=False)
        n, m = A.shape[0], P_T.shape[0]
        v_A = vertex_to_aggregate(P_T)
        cA, x = _f64(coords_A).reshape(m, dim), _f64(positions).reshape(n, dim)
        F = np.zeros((n, dim))
        _check(lib().ge_multilevel_forces(self.h, a.ref(), p.ref(), _ptr(v_A, _pi), _ptr(cA, _pd),
                                          _ptr(x, _pd), int(dim), C.byref(params), _ptr(F, _pd)))
        return F

    def galerkin(self, A, P_T, with_stats=False):
        """ge_galerkin: A_c = P_T A P_T^T (examples/embedder.cpp:213-216) -> scipy CSR (m x m)."""
        import scipy.sparse as sp
        a, pt = CsrView(A), CsrView(P_T, with_data=False)
        m = P_T.shape[0]
        cap = max(int(a.indptr[-1]), 1)
        ptr = np.zeros(m + 1, dtype=np.int32)
        idx = np.zeros(cap, dtype=np.int32)
        val = np.zeros(cap)
        nnz = C.c_int64()
        st = GalerkinStats()
        _check(lib().ge_galerkin(self.h, a.ref(), pt.ref(), _ptr(ptr, _pi), _ptr(idx, _pi), _ptr(val, _pd),
                                 C.c_int64(cap), C.byref(nnz), C.byref(st)))
        k = int(nnz.value)
        Ac = sp.csr_matrix((val[:k].copy(), idx[:k].copy(), ptr), shape=(m, m))
        if with_stats:
            return Ac, {f: getattr(st, f) for f, _ in st._fields_}
        return Ac

    def coarsen(self, A, coarsening_factor=0.25, min_coarse=64, max_levels=32, seed=0):
        """ge_coarsen: the hierarchy built on the device -> (As, P_Ts, stats) as scipy CSR, in the
        shape graphs.coarsen returns (As[0] is A)."""
        import scipy.sparse as sp
        A = sp.csr_matrix(A)
        a = CsrView(A)
        opt = CoarsenOptions()
        lib().ge_coarsen_options_default(C.byref(opt))
        opt.coarsening_factor, opt.min_coarse = float(coarsening_factor), int(min_coarse)
        opt.max_levels, opt.seed = int(max_levels), int(seed)
        st = CoarsenStats()
        h = C.c_void_p()
        _check(lib().ge_coarsen(self.h, a.ref(), C.byref(opt), C.byref(h), C.byref(st)))
        try:
            L = int(lib().ge_hierarchy_levels(h))
            As = [sp.csr_matrix((a.data, a.indices, a.indptr), shape=A.shape)]
            Ps = []
            for l in range(L):
                c = Csr()
                _check(lib().ge_hierarchy_aggregation(h, l, C.byref(c)))
                Ps.append(_csr_copy(c))
                _check(lib().ge_hierarchy_graph(h, l + 1, C.byref(c)))
                As.append(_csr_copy(c))
        finally:
            lib().ge_hierarchy_destroy(h)
        return As, Ps, {f: getattr(st, f) for f, _ in st._fields_}

    def largest_component(self, A):
        """ge_largest_component -> (B, vertices, components): B = A[vertices][:, vertices] as scipy CSR,
        vertices the kept original ids (ascending), components the number of components of A."""
        import scipy.sparse as sp
        a = CsrView(sp.csr_matrix(A))
        n = A.shape[0]
        cap = max(int(a.indptr[-1]), 1)
        vert = np.zeros(max(n, 1), dtype=np.int32)
        ptr = np.zeros(n + 1, dtype=np.int32)
        idx = np.zeros(cap, dtype=np.int32)
        val = np.zeros(cap)
        n_out, nnz, comps = C.c_int32(), C.c_int64(), C.c_int64()
        _check(lib().ge_largest_component(self.h, a.ref(), _ptr(vert, _pi), C.byref(n_out), _ptr(ptr, _pi),
                                          _ptr(idx, _pi), _ptr(val, _pd), C.c_int64(cap), C.byref(nnz),
                                          C.byref(comps)))
        k, e = int(n_out.value), int(nnz.value)
        B = sp.csr_matrix((val[:e].copy(), idx[:e].copy(), ptr[:k + 1].copy()), shape=(k, k))
        return B, vert[:k].copy(), int(comps.value)

    @staticmethod
    def _layout_options(coarsening_factor, min_coarse, max_levels, coarsen_seed, seed, precision,
                        coarse_iterations, level_iterations, verbose):
        copt = CoarsenOptions()
        lib().ge_coarsen_options_default(C.byref(copt))
        copt.coarsening_factor, copt.min_coarse = float(coarsening_factor), int(min_coarse)
        copt.max_levels, copt.seed = int(max_levels), int(coarsen_seed)
        eopt = EmbedOptions()
        lib().ge_embed_options_default(C.byref(eopt))
        eopt.seed, eopt.precision, eopt.verbose = int(seed), int(precision), int(verbose)
        eopt.coarse_iterations, eopt.level_iterations = int(coarse_iterations), int(level_iterations)
        return copt, eopt

    def layout(self, A, dim, coarsening_factor=0.25, min_coarse=64, max_levels=32, coarsen_seed=0, seed=0,
               largest_component=True, precision=GE_F64, coarse_iterations=100000, level_iterations=100,
               verbose=False):
        """ge_layout_graph: [largest component] -> ge_coarsen -> ge_embed in one call ->
        (coords [n x dim], vertices [n] original ids of the rows, stats)."""
        import scipy.sparse as sp
        a = CsrView(sp.csr_matrix(A))
        copt, eopt = self._layout_options(coarsening_factor, min_coarse, max_levels, coarsen_seed, seed, precision,
                                          coarse_iterations, level_iterations, verbose)
        n = A.shape[0]
        out = np.zeros((max(n, 1), dim))
        vert = np.zeros(max(n, 1), dtype=np.int32)
        n_out = C.c_int32()
        st = LayoutStats()
        _check(lib().ge_layout_graph(self.h, a.ref(), int(dim), int(bool(largest_component)), C.byref(copt),
                                     C.byref(eopt), _ptr(out, _pd), _ptr(vert, _pi), C.byref(n_out),
                                     C.byref(st)))
        k = int(n_out.value)
        return out[:k].copy(), vert[:k].copy(), _struct_dict(st)

    def graph_from_edges(self, n, src, dst, weights=None, symmetrize=True, keep_self_loops=False,
                         unit_weights=False):
        """ge_graph_from_edges: the CSR CooMatrix builds from the edges src[e] -> dst[e] (weights None:
        1.0) -> (scipy CSR n x n, stats)."""
        import scipy.sparse as sp
        el = EdgeList(n, src, dst, weights)
        opt = edges_options(symmetrize, keep_self_loops, unit_weights)
        cap = max(el.E * (2 if symmetrize else 1), 1)
        ptr = np.zeros(el.n + 1, dtype=np.int32)
        idx = np.empty(cap, dtype=np.int32)
        val = np.empty(cap)
        nnz = C.c_int64()
        st = EdgesStats()
        _check(lib().ge_graph_from_edges(self.h, *el.args(), C.byref(opt), _ptr(ptr, _pi), _ptr(idx, _pi),
                                         _ptr(val, _pd), C.c_int64(cap), C.byref(nnz), C.byref(st)))
        k = int(nnz.value)
        return sp.csr_matrix((val[:k], idx[:k], ptr), shape=(el.n, el.n)), _struct_dict(st)

    def layout_edges(self, n, src, dst, dim, weights=None, symmetrize=True, keep_self_loops=False,
                     unit_weights=False, coarsening_factor=0.25, min_coarse=64, max_levels=32, coarsen_seed=0,
                     seed=0, largest_component=True, precision=GE_F64, coarse_iterations=100000,
                     level_iterations=100, verbose=False):
        """ge_layout_edges: edge list -> graph -> [largest component] -> ge_coarsen -> ge_embed in one
        call -> (coords [k x dim], vertices [k] original ids of the rows, edges stats, layout stats)."""
        el = EdgeList(n, src, dst, weights)
        xopt = edges_options(symmetrize, keep_self_loops, unit_weights)
        copt, eopt = self._layout_options(coarsening_factor, min_coarse, max_levels, coarsen_seed, seed, precision,
                                          coarse_iterations, level_iterations, verbose)
        out = np.zeros((max(el.n, 1), dim))
        vert = np.zeros(max(el.n, 1), dtype=np.int32)
        n_out = C.c_int32()
        xs, st = EdgesStats(), LayoutStats()
        _check(lib().ge_layout_edges(self.h, *el.args(), C.byref(xopt), int(dim), int(bool(largest_component)),
                                     C.byref(copt), C.byref(eopt), _ptr(out, _pd), _ptr(vert, _pi),
                                     C.byref(n_out), C.byref(xs), C.byref(st)))
        k = int(n_out.value)
        return out[:k].copy(), vert[:k].copy(), _struct_dict(xs), _struct_dict(st)

    def flat_plan(self, A, dim, params, rows=None, symmetric=None):
        """rows=(r0, r1): ordered row-block plan; symmetric=(rank, world): that rank's plan of a
        symmetric multi-rank solve (see ge_flat_plan_create_symmetric)."""
        return FlatPlan(self, A, dim, params, rows, symmetric)


def symmetric_share(ld, rank, world):
    """ge_flat_symmetric_share -> [(row0, row1, tile_first, ntiles, tile_sym0)] (host only)."""
    L = lib()
    L.ge_flat_symmetric_share.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    nb = L.ge_flat_symmetric_share(int(ld), int(rank), int(world), 0, None)
    if nb < 0:
        raise ValueError("bad arguments")
    buf = np.zeros(max(nb, 1) * 5, dtype=np.int32)
    L.ge_flat_symmetric_share(int(ld), int(rank), int(world), nb, buf.ctypes.data_as(C.c_void_p))
    return [tuple(int(v) for v in buf[5 * i:5 * i + 5]) for i in range(nb)]


def symmetric_pass_share(ld, rank, world, npass, q):
    """ge_flat_symmetric_pass_share -> [(row0, row1, tile_first, ntiles, tile_sym0)] (host only)."""
    L = lib()
    L.ge_flat_symmetric_pass_share.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                C.c_int32, C.c_void_p]
    nb = L.ge_flat_symmetric_pass_share(int(ld), int(rank), int(world), int(npass), int(q), 0, None)
    if nb < 0:
        raise ValueError("bad arguments")
    buf = np.zeros(max(nb, 1) * 5, dtype=np.int32)
    L.ge_flat_symmetric_pass_share(int(ld), int(rank), int(world), int(npass), int(q), nb,
                                   buf.ctypes.data_as(C.c_void_p))
    return [tuple(int(v) for v in buf[5 * i:5 * i + 5]) for i in range(nb)]


def embed_aggregate_ranges(A, P_T, ndev):
    """ge_embed_aggregate_ranges -> (cuts[ndev + 1], ordered pairs per iteration) (host only)."""
    a, p = CsrView(A), CsrView(P_T, with_data=False)
    cuts = np.zeros(ndev + 1, dtype=np.int32)
    pairs = C.c_double()
    _check(lib().ge_embed_aggregate_ranges(a.ref(), p.ref(), int(ndev), _ptr(cuts, _pi), C.byref(pairs)))
    return cuts, pairs.value


def embed_aggregate_owners(A, P_T, ndev):
    """ge_embed_aggregate_owners -> (owner[m], ordered pairs per iteration) (host only)."""
    a, p = CsrView(A), CsrView(P_T, with_data=False)
    owner = np.zeros(max(P_T.shape[0], 1), dtype=np.int32)
    pairs = C.c_double()
    _check(lib().ge_embed_aggregate_owners(a.ref(), p.ref(), int(ndev), _ptr(owner, _pi), C.byref(pairs)))
    return owner[:P_T.shape[0]], pairs.value


class FlatPlan:
    """ge_flat_plan: device-resident flat solver for rows [r0, r1) of A."""

    def __init__(self, ctx, A, dim, params, rows=None, symmetric=None):
        self.ctx, self.n, self.dim = ctx, A.shape[0], dim
        self.rows = rows if rows is not None else (0, A.shape[0])
        a = CsrView(A)
        self.h = C.c_void_p()
        if symmetric is not None:
            rank, world = symmetric
            ld = ((max(self.n, 1) + 255) // 256) * 256
            R = ld // world
            self.rows = (min(self.n, rank * R), min(self.n, (rank + 1) * R))
            _check(lib().ge_flat_plan_create_symmetric(ctx.h, a.ref(), int(dim), C.byref(params),
                                                       int(rank), int(world), C.byref(self.h)))
        else:
            _check(lib().ge_flat_plan_create(ctx.h, a.ref(), int(dim), C.byref(params),
                                             int(self.rows[0]), int(self.rows[1]), C.byref(self.h)))
        self.symmetric = bool(lib().ge_flat_plan_is_symmetric(self.h))
        self.ld = int(lib().ge_flat_plan_ld(self.h))
        self.elem_size = int(lib().ge_flat_plan_elem_size(self.h))

    def close(self):
        if self.h:
            lib().ge_flat_plan_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def bind_coords(self, ptr0, ptr1):
        _check(lib().ge_flat_plan_bind_coords(self.h, C.c_void_p(ptr0), C.c_void_p(ptr1)))

    def upload(self, coords):
        x = _f64(coords).reshape(self.n, self.dim)
        _check(lib().ge_flat_plan_upload_coords(self.h, _ptr(x, _pd)))

    def download(self):
        out = np.zeros((self.n, self.dim))
        _check(lib().ge_flat_plan_download_coords(self.h, _ptr(out, _pd)))
        return out

    def download_forces(self):
        out = np.zeros((self.rows[1] - self.rows[0], self.dim))
        _check(lib().ge_flat_plan_download_forces(self.h, _ptr(out, _pd)))
        return out

    def cur_ptr(self):
        return lib().ge_flat_plan_cur_coords(self.h)

    def next_ptr(self):
        return lib().ge_flat_plan_next_coords(self.h)

    def launch_iteration(self):
        _check(lib().ge_flat_plan_launch_iteration(self.h))

    def launch_repulsion(self):
        _check(lib().ge_flat_plan_launch_repulsion(self.h))

    def launch_step(self):
        _check(lib().ge_flat_plan_launch_step(self.h))

    def pair_sums_ptr(self):
        return lib().ge_flat_plan_pair_sums(self.h)

    def bind_pair_sums(self, ptr):
        _check(lib().ge_flat_plan_bind_pair_sums(self.h, C.c_void_p(ptr)))

    def swap(self):
        lib().ge_flat_plan_swap(self.h)

    def iterate(self, iters):
        _check(lib().ge_flat_plan_iterate(self.h, int(iters)))

    def sync(self):
        _check(lib().ge_flat_plan_sync(self.h))

    def select_kernels(self, mask):
        lib().ge_flat_plan_select_kernels(self.h, int(mask))

    def profile(self, enable=True):
        lib().ge_flat_plan_profile(self.h, int(enable))

    def profile_get(self):
        rep, step = C.c_double(), C.c_double()
        nrep, nstep = C.c_int64(), C.c_int64()
        _check(lib().ge_flat_plan_profile_get(self.h, C.byref(rep), C.byref(nrep), C.byref(step),
                                              C.byref(nstep)))
        return dict(repulsion_ms=rep.value, repulsion_launches=nrep.value,
                    attract_step_ms=step.value, attract_step_launches=nstep.value)
