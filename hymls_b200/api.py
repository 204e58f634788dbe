"""ctypes binding of include/hymls_b200.h, shaped like the reference classes.

    HYMLS::Preconditioner(K, params, testVector)  -> Preconditioner(K, params, testvector)
        Initialize / Compute / ApplyInverse        (src/HYMLS_Preconditioner.hpp:98-254)
    HYMLS::Solver(K, P, params)::ApplyInverse(b,x) -> Solver(prec).ApplyInverse(b)
                                                    (src/HYMLS_BaseSolver.cpp:309-359)
`params` is either the XML text of a Teuchos ParameterList or a nested dict.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

HOST, DEVICE = 0, 1
MAP_OVERLAPPING, MAP_INTERIOR, MAP_SEPARATOR, MAP_VSUM = 0, 1, 2, 3


class HymlsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("hymls_b200 error %d: %s" % (code, msg))
        self.code = code


class _SolveInfo(C.Structure):
    _fields_ = [("iterations", C.c_int), ("converged", C.c_int), ("rel_residual", C.c_double),
                ("explicit_rel_residual", C.c_double), ("solve_seconds", C.c_double), ("history_len", C.c_int)]


class _Stats(C.Structure):
    _fields_ = [("num_initialize", C.c_int), ("num_compute", C.c_int), ("num_apply_inverse", C.c_int),
                ("time_initialize", C.c_double), ("time_compute", C.c_double), ("time_apply_inverse", C.c_double),
                ("n", C.c_int64), ("num_interior", C.c_int64), ("num_separator", C.c_int64), ("num_vsum", C.c_int64),
                ("num_subdomains", C.c_int64), ("num_blocks", C.c_int64), ("sum_nsd_sq", C.c_double),
                ("bytes_apply", C.c_double), ("flops_compute", C.c_double), ("bytes_a11_level0", C.c_double),
                ("kernel_launches", C.c_int64), ("device_bytes", C.c_double), ("sum_nsd_nb", C.c_double),
                ("bytes_a11_full_pass", C.c_double), ("ms_a11_lead", C.c_double), ("interior_couplings", C.c_int64),
                ("a11_split", C.c_int64), ("host_pipeline_chunks", C.c_int64), ("host_pipeline_state", C.c_int64),
                ("collective_calls", C.c_int64), ("collective_bytes", C.c_int64)]


def lib_path():
    return os.path.join(_HERE, "libhymls_b200.so")


def load_library():
    """Loads the CUDA library; fails loudly if it has not been built (no fallback)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError("hymls_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "or `make -C hymls_b200/csrc`; there is no CPU fallback" % path)
    lib = C.CDLL(path)
    P = C.POINTER
    vp, i64, dbl = C.c_void_p, C.c_int64, C.c_double
    lib.hymls_b200_last_error.restype = C.c_char_p
    lib.hymls_b200_version.restype = C.c_char_p
    lib.hymls_b200_create.argtypes = [C.c_char_p, P(vp)]
    lib.hymls_b200_destroy.argtypes = [vp]
    lib.hymls_b200_destroy.restype = None
    lib.hymls_b200_set_stream.argtypes = [vp, vp]
    lib.hymls_b200_comm_get_unique_id.argtypes = [vp]
    lib.hymls_b200_comm_init.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.hymls_b200_set_rank.argtypes = [vp, C.c_int, C.c_int]
    lib.hymls_b200_get_owned_subdomains.argtypes = [vp, C.c_int, vp, C.c_int]
    lib.hymls_b200_set_matrix_csr.argtypes = [vp, i64, vp, vp, vp, C.c_int]
    lib.hymls_b200_set_testvector.argtypes = [vp, vp]
    lib.hymls_b200_set_matrix_csr_dist.argtypes = [vp, i64, i64, vp, vp, vp, vp]
    lib.hymls_b200_set_parameters.argtypes = [vp, C.c_char_p]
    lib.hymls_b200_set_row_map.argtypes = [vp, i64, vp]
    lib.hymls_b200_apply_inverse_map.argtypes = [vp, vp, i64, vp, i64, C.c_int, C.c_int]
    lib.hymls_b200_apply_inverse_bordered_map.argtypes = [vp, vp, i64, vp, vp, i64, vp, C.c_int, C.c_int]
    lib.hymls_b200_set_testvector_dist.argtypes = [vp, i64, vp, vp]
    lib.hymls_b200_set_border_dist.argtypes = [vp, i64, vp, vp, vp, vp, C.c_int]
    lib.hymls_b200_initialize.argtypes = [vp]
    lib.hymls_b200_compute.argtypes = [vp]
    lib.hymls_b200_apply_inverse.argtypes = [vp, vp, i64, vp, i64, C.c_int, C.c_int]
    lib.hymls_b200_local_rows.argtypes = [vp, P(i64), P(i64)]
    lib.hymls_b200_owned_rows.argtypes = [vp, vp, i64]
    lib.hymls_b200_owned_rows.restype = i64
    lib.hymls_b200_apply_inverse_dist.argtypes = [vp, vp, vp, C.c_int]
    lib.hymls_b200_apply_inverse_bordered_dist.argtypes = [vp, vp, vp, vp, vp, C.c_int]
    lib.hymls_b200_border_size.argtypes = [vp]
    lib.hymls_b200_get_device.argtypes = [vp]
    lib.hymls_b200_set_border.argtypes = [vp, vp, vp, vp, C.c_int]
    lib.hymls_b200_apply_inverse_bordered.argtypes = [vp, vp, i64, vp, vp, i64, vp, C.c_int, C.c_int]
    lib.hymls_b200_apply_matrix.argtypes = [vp, vp, vp, C.c_int]
    lib.hymls_b200_solve.argtypes = [vp, vp, vp, C.c_int, C.c_uint64, P(_SolveInfo), vp, C.c_int]
    lib.hymls_b200_set_tolerance.argtypes = [vp, C.c_double]
    lib.hymls_b200_get_parameters_xml.argtypes = [vp, C.c_char_p, i64]
    lib.hymls_b200_get_parameters_xml.restype = i64
    lib.hymls_b200_num_levels.argtypes = [vp]
    lib.hymls_b200_num_subdomains.argtypes = [vp, C.c_int]
    lib.hymls_b200_get_interior.argtypes = [vp, C.c_int, C.c_int, vp, i64]
    lib.hymls_b200_get_interior.restype = i64
    lib.hymls_b200_get_groups.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, i64, P(i64)]
    lib.hymls_b200_get_map.argtypes = [vp, C.c_int, C.c_int, vp, i64]
    lib.hymls_b200_get_map.restype = i64
    lib.hymls_b200_pid_map.argtypes = [C.c_char_p, C.c_int, vp, C.c_int]
    lib.hymls_b200_get_stats.argtypes = [vp, P(_Stats)]
    lib.hymls_b200_time_apply.argtypes = [vp, C.c_int, P(dbl), P(dbl)]
    lib.hymls_b200_debug_copy.argtypes = [vp, C.c_int, C.c_char_p, vp, i64]
    lib.hymls_b200_debug_copy.restype = i64
    _LIB = lib
    return lib


def _check(lib, rc):
    if rc < 0:
        raise HymlsError(rc, lib.hymls_b200_last_error().decode())
    return rc


def _xml_escape(s):
    return (str(s).replace("&", "&amp;").replace("<", "&lt;").replace(">", "&gt;").replace('"', "&quot;"))


def params_to_xml(params, name="HYMLS"):
    """nested dict -> Teuchos ParameterList XML (bool/int/float/str leaves)."""
    if isinstance(params, str):
        return params
    out = ['<ParameterList name="%s">' % _xml_escape(name)]
    for k, v in params.items():
        if isinstance(v, dict):
            out.append(params_to_xml(v, k))
        elif isinstance(v, bool):
            out.append('<Parameter name="%s" type="bool" value="%s"/>' % (_xml_escape(k), "true" if v else "false"))
        elif isinstance(v, (int, np.integer)):
            out.append('<Parameter name="%s" type="int" value="%d"/>' % (_xml_escape(k), int(v)))
        elif isinstance(v, (float, np.floating)):
            out.append('<Parameter name="%s" type="double" value="%r"/>' % (_xml_escape(k), float(v)))
        else:
            out.append('<Parameter name="%s" type="string" value="%s"/>' % (_xml_escape(k), _xml_escape(v)))
    out.append("</ParameterList>")
    return "\n".join(out)


def pid_map(params, nprocs):
    """BasePartitioner::CreatePIDMap for `nprocs` ranks (src/HYMLS_BasePartitioner.cpp:361-586)."""
    lib = load_library()
    xml = params_to_xml(params).encode()
    n = _check(lib, lib.hymls_b200_pid_map(xml, nprocs, None, 0))
    out = np.zeros(n, dtype=np.int32)
    _check(lib, lib.hymls_b200_pid_map(xml, nprocs, out.ctypes.data, n))
    return out


def _ptr(a):
    """host numpy array or torch CUDA tensor -> (pointer, where)"""
    if isinstance(a, np.ndarray):
        return a.ctypes.data, HOST
    if hasattr(a, "data_ptr"):
        return a.data_ptr(), (DEVICE if a.is_cuda else HOST)
    raise TypeError("expected a numpy array or a torch tensor")


class Preconditioner:
    """HYMLS::Preconditioner : Ifpack_Preconditioner (src/HYMLS_Preconditioner.hpp:56-254)."""

    def __init__(self, K, params, testvector=None, cuda_stream=None, pattern_only=False):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.params_xml = params_to_xml(params)
        _check(self._lib, self._lib.hymls_b200_create(self.params_xml.encode(), C.byref(self._h)))
        if cuda_stream is not None:
            _check(self._lib, self._lib.hymls_b200_set_stream(self._h, C.c_void_p(cuda_stream)))
        self.n = 0
        if K is not None:
            self.SetMatrix(K, pattern_only=pattern_only)
        if testvector is not None:
            tv = np.ascontiguousarray(testvector, dtype=np.float64)
            _check(self._lib, self._lib.hymls_b200_set_testvector(self._h, tv.ctypes.data))

    def __del__(self):
        try:
            if self._h:
                self._lib.hymls_b200_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    # -- Preconditioner::SetMatrix (:250-254): scipy CSR (host) or (rowptr, colidx, values) arrays/tensors
    def SetMatrix(self, K, pattern_only=False):
        if isinstance(K, tuple):
            rowptr, colidx, values = K
            n = len(rowptr) - 1
            p_rp, w1 = _ptr(rowptr)
            p_ci, w2 = _ptr(colidx)
            p_v, w3 = _ptr(values)
            assert w1 == w2 == w3
            self._keep = (rowptr, colidx, values)
            _check(self._lib, self._lib.hymls_b200_set_matrix_csr(self._h, n, p_rp, p_ci, p_v, w1))
        else:
            K = K.tocsr()
            K.sort_indices()
            n = K.shape[0]
            rp = np.ascontiguousarray(K.indptr, dtype=np.int64)
            ci = np.ascontiguousarray(K.indices, dtype=np.int32)
            v = np.ascontiguousarray(K.data, dtype=np.float64)
            _check(self._lib, self._lib.hymls_b200_set_matrix_csr(
                self._h, n, rp.ctypes.data, ci.ctypes.data, None if pattern_only else v.ctypes.data, HOST))
        self.n = n
        return 0

    # -- distributed caller (one MPI rank per GPU): rows / vectors on the caller's map --------------------
    def SetMatrixDist(self, n_global, row_gids, K_local, pattern_only=False):
        """this rank's rows (scipy CSR with GLOBAL column ids, row i <-> row_gids[i]); collective"""
        K = K_local.tocsr()
        g = np.ascontiguousarray(row_gids, dtype=np.int64)
        rp = np.ascontiguousarray(K.indptr, dtype=np.int64)
        ci = np.ascontiguousarray(K.indices, dtype=np.int64)
        v = np.ascontiguousarray(K.data, dtype=np.float64)
        _check(self._lib, self._lib.hymls_b200_set_matrix_csr_dist(
            self._h, n_global, len(g), g.ctypes.data, rp.ctypes.data, ci.ctypes.data,
            None if pattern_only else v.ctypes.data))
        self.n = n_global
        return 0

    def SetParameters(self, params):
        return _check(self._lib, self._lib.hymls_b200_set_parameters(self._h, params_to_xml(params).encode()))

    def SetTestVectorDist(self, row_gids, tv_local):
        g = np.ascontiguousarray(row_gids, dtype=np.int64)
        t = np.ascontiguousarray(tv_local, dtype=np.float64)
        return _check(self._lib, self._lib.hymls_b200_set_testvector_dist(self._h, len(g), g.ctypes.data, t.ctypes.data))

    def SetRowMap(self, row_gids):
        g = np.ascontiguousarray(row_gids, dtype=np.int64)
        self._nlocal = len(g)
        return _check(self._lib, self._lib.hymls_b200_set_row_map(self._h, len(g), g.ctypes.data))

    def ApplyInverseMap(self, B_local):
        """vectors on the map given to SetRowMap (numpy, host; n_local or n_local x nvec)"""
        Bc = np.asfortranarray(np.asarray(B_local, dtype=np.float64).reshape(self._nlocal, -1))
        Xc = np.zeros_like(Bc, order="F")
        _check(self._lib, self._lib.hymls_b200_apply_inverse_map(self._h, Bc.ctypes.data, self._nlocal, Xc.ctypes.data,
                                                                  self._nlocal, Bc.shape[1], HOST))
        return Xc.reshape(np.shape(B_local))

    # -- multi-GPU (one process per GPU) -------------------------------------------------------------
    @staticmethod
    def CommUniqueId():
        lib = load_library()
        buf = (C.c_char * 128)()
        _check(lib, lib.hymls_b200_comm_get_unique_id(buf))
        return bytes(buf)

    def CommInit(self, unique_id, rank, nranks):
        buf = (C.c_char * 128).from_buffer_copy(unique_id)
        return _check(self._lib, self._lib.hymls_b200_comm_init(self._h, buf, rank, nranks))

    def SetRank(self, rank, nranks):
        return _check(self._lib, self._lib.hymls_b200_set_rank(self._h, rank, nranks))

    def OwnedSubdomains(self, level=0):
        n = _check(self._lib, self._lib.hymls_b200_get_owned_subdomains(self._h, level, None, 0))
        out = np.zeros(n, dtype=np.int32)
        if n:
            _check(self._lib, self._lib.hymls_b200_get_owned_subdomains(self._h, level, out.ctypes.data, n))
        return out

    def Initialize(self):
        return _check(self._lib, self._lib.hymls_b200_initialize(self._h))

    def Compute(self):
        rc = _check(self._lib, self._lib.hymls_b200_compute(self._h))
        # "Visualize Solver" (src/HYMLS_Preconditioner.cpp:510-514): MATLAB file with the partitioning
        if 'name="Visualize Solver" type="bool" value="true"' in self.params_xml:
            self.Visualize("hid_data.m")
        return rc

    def Visualize(self, mfilename, no_recurse=False):
        """Preconditioner::Visualize (src/HYMLS_Preconditioner.cpp:753-779)"""
        from . import io
        io.visualize(self, mfilename, no_recurse)

    def ApplyInverse(self, B, X=None):
        """X = P^-1 B.  numpy (host) or torch CUDA tensors (device, column major: shape (nvec, n) contiguous
        or 1-D)."""
        if isinstance(B, np.ndarray):
            Bc = np.asfortranarray(B.reshape(self.n, -1), dtype=np.float64)
            nvec = Bc.shape[1]
            Xc = np.zeros_like(Bc, order="F")
            _check(self._lib, self._lib.hymls_b200_apply_inverse(self._h, Bc.ctypes.data, self.n, Xc.ctypes.data,
                                                                  self.n, nvec, HOST))
            return Xc.reshape(B.shape) if B.ndim == 1 else Xc
        import torch
        assert B.is_cuda and B.dtype == torch.float64 and B.is_contiguous()
        nvec = 1 if B.dim() == 1 else B.shape[0]
        if X is None:
            X = torch.empty_like(B)
        _check(self._lib, self._lib.hymls_b200_apply_inverse(self._h, B.data_ptr(), self.n, X.data_ptr(), self.n,
                                                              nvec, DEVICE))
        return X

    def LocalRows(self):
        a, b = C.c_int64(), C.c_int64()
        _check(self._lib, self._lib.hymls_b200_local_rows(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def OwnedRows(self):
        """rows (GIDs, ascending) this rank owns: interiors of its subdomains + the separator groups it owns"""
        n = int(self._lib.hymls_b200_owned_rows(self._h, None, 0))
        _check(self._lib, n)
        out = np.zeros(n, dtype=np.int64)
        _check(self._lib, int(self._lib.hymls_b200_owned_rows(self._h, out.ctypes.data, n)))
        return out

    def ApplyInverseDist(self, b_local):
        """distributed-vector ApplyInverse: the rows of OwnedRows() in, the same rows out (numpy: host buffers,
        torch CUDA tensors: device buffers)"""
        if isinstance(b_local, np.ndarray):
            bl = np.ascontiguousarray(b_local, dtype=np.float64)
            xl = np.zeros_like(bl)
            _check(self._lib, self._lib.hymls_b200_apply_inverse_dist(self._h, bl.ctypes.data, xl.ctypes.data, HOST))
            return xl
        import torch
        xl = torch.empty_like(b_local)
        _check(self._lib, self._lib.hymls_b200_apply_inverse_dist(self._h, b_local.data_ptr(), xl.data_ptr(), DEVICE))
        return xl

    def Apply(self, X, Y):  # Preconditioner::Apply returns -1 (:122-123)
        return -1

    def SetUseTranspose(self, flag):  # returns -1 (:162-166)
        return -1

    def SetBorder(self, V, W=None, Cm=None):
        """BorderedOperator::SetBorder(V, W, C) (src/HYMLS_Preconditioner.cpp:844-918); V=None removes it.
        Compute() has to be called afterwards."""
        if V is None:
            return _check(self._lib, self._lib.hymls_b200_set_border(self._h, None, None, None, 0))
        Vc = np.asfortranarray(np.asarray(V, dtype=np.float64).reshape(self.n, -1))
        m = Vc.shape[1]
        Wc = None if W is None else np.asfortranarray(np.asarray(W, dtype=np.float64).reshape(self.n, -1))
        Cc = None if Cm is None else np.asfortranarray(np.asarray(Cm, dtype=np.float64).reshape(m, m))
        return _check(self._lib, self._lib.hymls_b200_set_border(
            self._h, Vc.ctypes.data, None if Wc is None else Wc.ctypes.data,
            None if Cc is None else Cc.ctypes.data, m))

    def BorderSize(self):
        """m of the border set with SetBorder or hymls_b200_set_border_dist (0: none)"""
        return self._lib.hymls_b200_border_size(self._h)

    def ApplyInverseBordered(self, B, T):
        """[X; S] = [K V; W' C]^-1 [B; T] approximately (BorderedOperator::ApplyInverse of the preconditioner,
        src/HYMLS_Preconditioner.cpp:930-1070).  numpy, host: B is n (x nvec), T is m (x nvec)."""
        Bc = np.asfortranarray(np.asarray(B, dtype=np.float64).reshape(self.n, -1))
        nvec = Bc.shape[1]
        Tc = np.asfortranarray(np.asarray(T, dtype=np.float64).reshape(-1, nvec))
        Xc = np.zeros_like(Bc, order="F")
        Sc = np.zeros_like(Tc, order="F")
        _check(self._lib, self._lib.hymls_b200_apply_inverse_bordered(
            self._h, Bc.ctypes.data, self.n, Tc.ctypes.data, Xc.ctypes.data, self.n, Sc.ctypes.data, nvec, HOST))
        return Xc, Sc

    def ApplyInverseBorderedDist(self, b_local, T):
        """[x; S] = [K V; W' C]^-1 [b; T] on the rows of OwnedRows(): b_local holds those rows, T (length m, the same on
        every rank) the border right-hand side; returns (x_local, S), S bitwise equal on every rank.  Both numpy
        (host buffers) or both 1-D torch CUDA tensors on the handle's device (device buffers), float64 and
        contiguous."""
        m = self.BorderSize()
        if m == 0:
            raise ValueError("ApplyInverseBorderedDist: no border set (SetBorder)")
        nown = int(self._lib.hymls_b200_owned_rows(self._h, None, 0))
        _check(self._lib, nown)

        def need(ok, what):
            if not ok:
                raise ValueError("ApplyInverseBorderedDist: " + what)

        if isinstance(b_local, np.ndarray):
            need(isinstance(T, np.ndarray), "b_local is a numpy array, so T must be one")
            for name, a, ln in (("b_local", b_local, nown), ("T", T, m)):
                need(a.dtype == np.float64, "%s must be float64" % name)
                need(a.ndim == 1 and a.shape[0] == ln, "%s must be 1-D of length %d" % (name, ln))
                need(a.flags.c_contiguous, "%s must be contiguous" % name)
            xl = np.zeros(nown)
            S = np.zeros(m)
            where = HOST
        else:
            import torch
            need(isinstance(b_local, torch.Tensor) and isinstance(T, torch.Tensor), "expected numpy arrays or torch tensors")
            dev = _check(self._lib, self._lib.hymls_b200_get_device(self._h))
            for name, a, ln in (("b_local", b_local, nown), ("T", T, m)):
                need(a.is_cuda and a.device.index == dev, "%s must be a CUDA tensor on cuda:%d, the handle's device"
                     % (name, dev))
                need(a.dtype == torch.float64, "%s must be float64" % name)
                need(a.dim() == 1 and a.shape[0] == ln, "%s must be 1-D of length %d" % (name, ln))
                need(a.is_contiguous(), "%s must be contiguous" % name)
            xl = torch.empty_like(b_local)
            S = torch.empty_like(T)
            where = DEVICE
        p = lambda a: a.ctypes.data if where == HOST else a.data_ptr()  # noqa: E731
        _check(self._lib, self._lib.hymls_b200_apply_inverse_bordered_dist(self._h, p(b_local), p(T), p(xl), p(S),
                                                                            where))
        return xl, S

    def ApplyMatrix(self, x):
        if isinstance(x, np.ndarray):
            xc = np.ascontiguousarray(x, dtype=np.float64)
            y = np.zeros_like(xc)
            _check(self._lib, self._lib.hymls_b200_apply_matrix(self._h, xc.ctypes.data, y.ctypes.data, HOST))
            return y
        import torch
        y = torch.empty_like(x)
        _check(self._lib, self._lib.hymls_b200_apply_matrix(self._h, x.data_ptr(), y.data_ptr(), DEVICE))
        return y

    def GetParametersXml(self):
        """The list with the defaults written back (the reference's 'Store Final Parameter List')."""
        n = int(self._lib.hymls_b200_get_parameters_xml(self._h, None, 0))
        _check(self._lib, n)
        buf = C.create_string_buffer(n + 1)
        self._lib.hymls_b200_get_parameters_xml(self._h, buf, n + 1)
        return buf.value.decode()

    # -- index maps --------------------------------------------------------------------------------
    def NumLevels(self):
        return self._lib.hymls_b200_num_levels(self._h)

    def NumMySubdomains(self, level=0):
        return _check(self._lib, self._lib.hymls_b200_num_subdomains(self._h, level))

    def GetInteriorGroup(self, sd, level=0):
        n = self._lib.hymls_b200_get_interior(self._h, level, sd, None, 0)
        _check(self._lib, int(n))
        out = np.zeros(n, dtype=np.int64)
        self._lib.hymls_b200_get_interior(self._h, level, sd, out.ctypes.data, n)
        return out

    def GetSeparatorGroups(self, sd, level=0):
        """[(type, gids)] in the reference's order (HierarchicalMap::GetSeparatorGroups)."""
        tot = C.c_int64()
        ng = _check(self._lib, self._lib.hymls_b200_get_groups(self._h, level, sd, None, None, None, 0, C.byref(tot)))
        ptr = np.zeros(ng + 1, dtype=np.int64)
        types = np.zeros(ng, dtype=np.int32)
        gids = np.zeros(tot.value, dtype=np.int64)
        _check(self._lib, self._lib.hymls_b200_get_groups(self._h, level, sd, ptr.ctypes.data, types.ctypes.data,
                                                           gids.ctypes.data, tot.value, C.byref(tot)))
        return [(int(types[g]), gids[ptr[g]:ptr[g + 1]]) for g in range(ng)]

    def GetMap(self, which, level=0):
        n = self._lib.hymls_b200_get_map(self._h, level, which, None, 0)
        _check(self._lib, int(n))
        out = np.zeros(n, dtype=np.int64)
        self._lib.hymls_b200_get_map(self._h, level, which, out.ctypes.data, n)
        return out

    def DebugArray(self, name, level=0):
        n = self._lib.hymls_b200_debug_copy(self._h, level, name.encode(), None, 0)
        _check(self._lib, int(n))
        out = np.zeros(n)
        if n:
            _check(self._lib, int(self._lib.hymls_b200_debug_copy(self._h, level, name.encode(), out.ctypes.data, n)))
        return out

    def Stats(self):
        st = _Stats()
        _check(self._lib, self._lib.hymls_b200_get_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in _Stats._fields_}

    def TimeApply(self, reps=20):
        a, b = C.c_double(), C.c_double()
        _check(self._lib, self._lib.hymls_b200_time_apply(self._h, reps, C.byref(a), C.byref(b)))
        return a.value, b.value


class Solver:
    """HYMLS::Solver(K, P, params): Krylov solve with the preconditioner (src/HYMLS_Solver.cpp:22-51,148-152).
    The "Solver" sublist is the one of the parameter list the preconditioner was created with."""

    def __init__(self, prec):
        self.prec = prec
        self.num_iter = 0
        self.info = None
        self.history = None

    def ApplyInverse(self, b, x=None, seed=43, history_cap=2048):
        P = self.prec
        lib = P._lib
        info = _SolveInfo()
        hist = np.zeros(history_cap)
        if isinstance(b, np.ndarray):
            bc = np.ascontiguousarray(b, dtype=np.float64)
            xc = np.zeros_like(bc) if x is None else np.ascontiguousarray(x, dtype=np.float64)
            _check(lib, lib.hymls_b200_solve(P._h, bc.ctypes.data, xc.ctypes.data, HOST, seed, C.byref(info),
                                             hist.ctypes.data, history_cap))
        else:
            import torch
            xc = torch.zeros_like(b) if x is None else x
            _check(lib, lib.hymls_b200_solve(P._h, b.data_ptr(), xc.data_ptr(), DEVICE, seed, C.byref(info),
                                             hist.ctypes.data, history_cap))
        self.num_iter = info.iterations
        self.info = {k: getattr(info, k) for k, _ in _SolveInfo._fields_}
        self.history = hist[:min(info.history_len, history_cap)].copy()
        return xc

    def getNumIter(self):
        return self.num_iter

    def SetTolerance(self, tol):
        """BaseSolver::SetTolerance: overrides "Convergence Tolerance" for the following solves (NOX does this)."""
        return _check(self.prec._lib, self.prec._lib.hymls_b200_set_tolerance(self.prec._h, float(tol)))
