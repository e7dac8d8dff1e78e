"""The ``harmony`` class: Python mirror of the reference's Rcpp module class
(/root/reference/src/harmony.cpp:672-709 — same method and field names, same shapes), implemented
by calls into the C ABI of include/harmony_b200.h.  This is what the reference's R code would hold
as ``harmonyObj`` (R/ui.R:269); the parity tests drive it exactly like the reference's testthat files.

Shapes follow R (column-major, cells are columns): ``obj.R`` is [K, N], ``obj.getZcorr()`` [d, N],
``obj.Y`` [d, K], ``obj.O`` / ``obj.E`` [K, B].  They are Fortran-ordered views of the buffers the
C ABI fills, i.e. the bytes an R numeric matrix would hold.
"""
import ctypes
import sys
import warnings

import numpy as np

from . import _lib

FIELD = {"Z_corr": 0, "Z_orig": 1, "R": 2, "Y": 3, "O": 4, "E": 5, "W": 6, "Pr_b": 7, "theta": 8, "sigma": 9,
         "lambda_mat": 10, "lambda": 11}
SCALAR = {"N": 0, "B": 1, "K": 2, "d": 3, "C": 4, "alpha": 5, "max_iter_kmeans": 6, "block_size": 7,
          "epsilon_kmeans": 8, "epsilon_harmony": 9, "N_local": 10, "lambda_estimation": 11, "window_size": 12,
          "legacy_centroid_step": 13, "kernel_set": 14, "device": 15}
TRACE = {"objective_kmeans": 0, "objective_kmeans_dist": 1, "objective_kmeans_entropy": 2,
         "objective_kmeans_cross": 3, "objective_harmony": 4, "kmeans_rounds": 5}
_INT_SCALARS = ("N", "B", "K", "d", "C", "max_iter_kmeans", "N_local", "window_size", "legacy_centroid_step", "kernel_set",
                "device")
HB_F32, HB_F64 = 0, 1   # enum hb_dtype


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class HarmonyError(RuntimeError):
    pass


def torch_of(x):
    """The torch module if ``x`` is a ``torch.Tensor``, else None.  Never imports torch: a caller that passes numpy
    arrays does not pay for it, and a tensor cannot exist unless torch was imported already."""
    torch = sys.modules.get("torch")
    return torch if torch is not None and isinstance(x, torch.Tensor) else None


def tensor_abi_args(Z, n):
    """(dtype code, cell stride, PC stride, d) of hb_setup_device for a 2-D float tensor ``Z`` of ``n`` cells, given as
    [n, d] or [d, n] (the same orientation rule as numpy input), any strides; strides are in elements."""
    torch = torch_of(Z)
    if Z.dim() != 2:
        raise ValueError(f"Z must be a 2-D tensor (cells x PCs or PCs x cells), not {Z.dim()}-D")
    codes = {torch.float32: HB_F32, torch.float64: HB_F64}
    if Z.dtype not in codes:
        raise TypeError(f"Z must be float32 or float64, not {Z.dtype}")
    if Z.shape[0] != n and Z.shape[1] == n:
        Z = Z.T
    if Z.shape[0] != n:
        raise ValueError("number of cells in Z and Phi differ")
    return codes[Z.dtype], int(Z.stride(0)), int(Z.stride(1)), int(Z.shape[1])


def _setup_params(sigma, theta, lambda_, K, B_vec):
    """Host-side scalars of harmony::setup as the C ABI takes them: (B_vec, K, sigma, theta, lambda or None)."""
    B_vec = np.ascontiguousarray(np.atleast_1d(B_vec), dtype=np.int32)
    K = int(K)
    sigma = np.ascontiguousarray(np.broadcast_to(np.asarray(sigma, dtype=np.float64), (K,)))
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    if len(theta) != int(B_vec.sum()):
        raise ValueError("theta must hold one value per covariate level")
    lam = None
    if lambda_ is not None and not (np.ndim(lambda_) == 0 and lambda_ == -1):
        lam = np.ascontiguousarray(np.atleast_1d(lambda_), dtype=np.float64)
        if len(lam) == 1 and lam[0] == -1:
            lam = None
        elif len(lam) != int(B_vec.sum()) + 1:
            raise ValueError("lambda must hold B+1 values")
    return B_vec, K, sigma, theta, lam


class harmony:
    """``new(harmony)`` — an opaque device-resident model; see module docstring."""

    def __init__(self, device=None, comm=None):
        object.__setattr__(self, "_h", None)
        L = _lib.lib()
        h = ctypes.c_void_p()
        st = L.hb_create(ctypes.byref(h), -1 if device is None else int(device))
        if st != 0 or not h:
            raise HarmonyError("hb_create failed: no usable CUDA device (harmony_b200 has no CPU fallback)")
        object.__setattr__(self, "_L", L)
        object.__setattr__(self, "_h", h)
        object.__setattr__(self, "_injected_orders", None)
        if comm is not None:
            self._init_comm(comm)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._L.hb_destroy(h)
            object.__setattr__(self, "_h", None)

    # ---- plumbing -------------------------------------------------------------------------------
    def _check(self, st):
        self._drain_warnings()
        if st != 0:
            raise HarmonyError(self._L.hb_last_error(self._h).decode())

    def _drain_warnings(self):
        buf = ctypes.create_string_buffer(512)
        while self._L.hb_pop_warning(self._h, buf, 512):
            warnings.warn(buf.value.decode())

    def _init_comm(self, comm):
        """comm = (rank, world_size, id_bytes or None, N_global, cell_offset); see harmony_b200.dist.
        ``id_bytes = None`` shares the process-wide communicator an earlier object created."""
        rank, world, uid, n_global, offset = comm
        self._check(self._L.hb_comm_init(self._h, int(rank), int(world), None if uid is None else bytes(uid)))
        self._check(self._L.hb_set_shard(self._h, int(n_global), int(offset)))

    def _scalar(self, name):
        v = ctypes.c_double()
        if self._L.hb_get_scalar(self._h, SCALAR[name], ctypes.byref(v)) != 0:
            raise HarmonyError(f"no scalar {name}")
        return int(v.value) if name in _INT_SCALARS else float(v.value)

    def _field(self, name, shape):
        n = self._L.hb_field_size(self._h, FIELD[name])
        out = np.empty(int(n), dtype=np.float64)
        self._check(self._L.hb_get_field(self._h, FIELD[name], _ptr(out)))
        return out.reshape(shape, order="F")

    # ---- methods of the Rcpp module (harmony.cpp:697-707) --------------------------------------
    def setup(self, Z, Phi, sigma, theta, lambda_, alpha, max_iter_kmeans, epsilon_kmeans, epsilon_harmony, K,
              block_size, B_vec, batch_proportion_cutoff, verbose=False):
        """harmony::setup (harmony.h:25-30).  ``Z``: [N, d] C-order (== the d x N column-major matrix
        of the reference) or [d, N] F-order; ``Phi``: the row-index slot of the B x N design matrix,
        int array [N, C]; ``lambda_``: B+1 values or None / -1 for automatic estimation.

        ``Z`` may also be a CUDA tensor (float32 / float64, [N, d] or [d, N], any strides) on this object's device;
        ``Phi`` is then a numpy array or a CUDA integer tensor.  Both are read on the current CUDA stream and nothing
        is copied through the host; the object ends in the state numpy input with the same values gives."""
        torch = torch_of(Z)
        if torch is not None and Z.is_cuda:
            return self._setup_device(torch, Z, Phi, sigma, theta, lambda_, alpha, max_iter_kmeans, epsilon_kmeans,
                                      epsilon_harmony, K, block_size, B_vec, batch_proportion_cutoff, verbose)
        Z = np.asarray(Z)
        phi_i = np.ascontiguousarray(Phi, dtype=np.int32)
        if phi_i.ndim == 1:
            phi_i = phi_i.reshape(-1, 1)
        n = phi_i.shape[0]
        if Z.ndim != 2:
            raise ValueError("Z must be a matrix")
        if Z.shape[0] != n and Z.shape[1] == n:
            Z = Z.T                                   # d x N given: its transpose view is the same memory order
        Z = np.ascontiguousarray(Z, dtype=np.float64)
        if Z.shape[0] != n:
            raise ValueError("number of cells in Z and Phi differ")
        B_vec, K, sigma, theta, lam = _setup_params(sigma, theta, lambda_, K, B_vec)
        self._check(self._L.hb_setup(self._h, _ptr(Z), Z.shape[1], n, _ptr(phi_i), _ptr(B_vec), len(B_vec),
                                     _ptr(sigma), _ptr(theta), None if lam is None else _ptr(lam), float(alpha),
                                     int(max_iter_kmeans), float(epsilon_kmeans), float(epsilon_harmony), K,
                                     float(block_size), float(batch_proportion_cutoff), int(bool(verbose))))

    def _setup_device(self, torch, Z, Phi, sigma, theta, lambda_, alpha, max_iter_kmeans, epsilon_kmeans,
                      epsilon_harmony, K, block_size, B_vec, batch_proportion_cutoff, verbose):
        dev = torch.device("cuda", self._scalar("device"))
        if Z.device != dev:
            raise ValueError(f"Z is on {Z.device}, this harmony object on {dev}")
        if torch_of(Phi) is not None:
            if Phi.is_cuda and Phi.device != dev:
                raise ValueError(f"Phi is on {Phi.device}, this harmony object on {dev}")
            if Phi.dtype.is_floating_point or Phi.dtype.is_complex or Phi.dtype == torch.bool:
                raise TypeError(f"Phi must hold integer level rows, not {Phi.dtype}")
            phi = Phi.to(device=dev, dtype=torch.int32)
        else:
            phi = torch.from_numpy(np.ascontiguousarray(Phi, dtype=np.int32)).to(dev)
        if phi.dim() == 1:
            phi = phi.reshape(-1, 1)
        phi = phi.contiguous()
        n = phi.shape[0]
        code, cell_stride, pc_stride, d = tensor_abi_args(Z, n)
        B_vec, K, sigma, theta, lam = _setup_params(sigma, theta, lambda_, K, B_vec)
        self._check(self._L.hb_setup_device(
            self._h, Z.data_ptr(), code, cell_stride, pc_stride, d, n, phi.data_ptr(), _ptr(B_vec), len(B_vec),
            _ptr(sigma), _ptr(theta), None if lam is None else _ptr(lam), float(alpha), int(max_iter_kmeans),
            float(epsilon_kmeans), float(epsilon_harmony), K, float(block_size), float(batch_proportion_cutoff),
            int(bool(verbose)), torch.cuda.current_stream(dev).cuda_stream))

    def to_torch(self, field="Z_corr", dtype=None, out=None):
        """A per-cell field as a CUDA tensor on this object's device, cells as rows: ``"Z_corr"`` / ``"Z_orig"``
        [N_local, d], ``"R"`` [N_local, K]; float32 unless ``dtype`` (float32 / float64) says otherwise.  ``out``: a
        preallocated tensor of that shape whose rows may be strided (e.g. a column slice of a wider tensor).  Ordered on
        the current CUDA stream without a host synchronisation; values are those of getZcorr() / getZorig() / R."""
        import torch
        cols = {"Z_corr": "d", "Z_orig": "d", "R": "K"}
        if field not in cols:
            raise ValueError(f"field must be one of {sorted(cols)}, not {field!r}")
        dev = torch.device("cuda", self._scalar("device"))
        shape = (self._scalar("N_local"), self._scalar(cols[field]))
        if out is None:
            out = torch.empty(shape, dtype=torch.float32 if dtype is None else dtype, device=dev)
        elif torch_of(out) is None or tuple(out.shape) != shape or out.device != dev or \
                (out.stride(1) != 1 and shape[1] > 1) or (dtype is not None and out.dtype != dtype):
            raise ValueError(f"out must be a {dtype or 'float'} tensor of shape {shape} on {dev} with unit column stride")
        codes = {torch.float32: HB_F32, torch.float64: HB_F64}
        if out.dtype not in codes:
            raise TypeError(f"to_torch writes float32 or float64, not {out.dtype}")
        ld = out.stride(0) if shape[0] > 1 else shape[1]
        self._check(self._L.hb_get_field_device(self._h, FIELD[field], out.data_ptr(), codes[out.dtype], ld,
                                                torch.cuda.current_stream(dev).cuda_stream))
        return out

    def debug_sort_perm(self):
        """Test hook: the tuple-sort permutation (position -> local cell)."""
        out = np.empty(self._scalar("N_local"), dtype=np.int32)
        if self._L.hb_debug_sort_perm(self._h, _ptr(out)) != 0:
            raise HarmonyError("hb_debug_sort_perm failed (setup has not run?)")
        return out
    def set_seed(self, seed):
        self._check(self._L.hb_set_seed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF))

    def init_cluster_cpp(self, Y0=None):
        """harmony::init_cluster_cpp.  ``Y0`` ([d, K] like ``obj.Y`` or [K, d] C-order) injects the
        k-means centroids (what kmeans_centers returns, harmony.cpp:133)."""
        if Y0 is None:
            self._check(self._L.hb_init_cluster(self._h, None))
            return
        K, d = self._scalar("K"), self._scalar("d")
        if K == 0:                                    # setup has not run: let the library report it
            self._check(self._L.hb_init_cluster(self._h, None))
        Y0 = np.asarray(Y0, dtype=np.float64)
        if Y0.shape == (d, K) and not (K == d and Y0.flags.c_contiguous):
            Y0 = Y0.T
        Y0 = np.ascontiguousarray(Y0)
        if Y0.shape != (K, d):
            raise ValueError("Y0 must be d x K")
        self._check(self._L.hb_init_cluster(self._h, _ptr(Y0)))

    def set_abort_callback(self, fn):
        """Progress::check_abort of the reference (harmony.cpp:233, 355): ``fn()`` is polled before the clustering
        rounds of every cluster_cpp call (and between them); a true value makes cluster_cpp return -1, which
        harmonize() turns into "terminated by user" (R/utils.R:27-29).  ``None`` removes the callback."""
        import ctypes
        if fn is None:
            self._abort_cb = None
            self._check(self._L.hb_set_abort_callback(self._h, None, None))
            return
        proto = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p)
        self._abort_cb = proto(lambda _user: 1 if fn() else 0)   # keep the trampoline alive with the object
        self._check(self._L.hb_set_abort_callback(self._h, ctypes.cast(self._abort_cb, ctypes.c_void_p), None))

    def cluster_cpp(self, update_orders=None):
        """harmony::cluster_cpp -> 0 / -1 (aborted).  ``update_orders``: [max_iter_kmeans, N] int64,
        row t = the shuffled update order of the t-th update_R call (harmony.cpp:272-273)."""
        if update_orders is None:
            st = self._L.hb_cluster(self._h, None)
        else:
            T, N = self._scalar("max_iter_kmeans"), self._scalar("N")
            uo = np.ascontiguousarray(update_orders, dtype=np.int64).reshape(-1, N)
            if uo.shape[0] < T:
                raise ValueError("need one update order per clustering round")
            st = self._L.hb_cluster(self._h, _ptr(uo))
        if st == -1:
            return -1
        self._check(st)
        return 0

    def moe_correct_ridge_cpp(self):
        self._check(self._L.hb_moe_correct_ridge(self._h))

    def check_convergence(self, type_):
        r = self._L.hb_check_convergence(self._h, int(type_))
        if r < 0:
            raise HarmonyError(self._L.hb_last_error(self._h).decode())
        return bool(r)

    def compute_objective(self):
        self._check(self._L.hb_compute_objective(self._h))

    def getZcorr(self):
        return self._field("Z_corr", (self._scalar("d"), self._scalar("N_local")))

    def getZorig(self):
        return self._field("Z_orig", (self._scalar("d"), self._scalar("N_local")))

    def getR(self):
        return self._field("R", (self._scalar("K"), self._scalar("N_local")))

    def getCentroids(self):
        return self._field("Y", (self._scalar("d"), self._scalar("K")))

    def getLambda(self):
        return self._field("lambda_mat", (self._scalar("K"), self._scalar("B") + 1))

    # ---- fields of the Rcpp module (harmony.cpp:675-696) ---------------------------------------
    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        if name in ("N", "B", "K", "d", "alpha", "max_iter_kmeans", "legacy_centroid_step", "kernel_set"):
            return self._scalar(name)
        if name == "R":
            return self.getR()
        if name == "Y":
            return self.getCentroids()
        if name in ("O", "E"):
            return self._field(name, (self._scalar("K"), self._scalar("B")))
        if name == "W":
            return self._field("W", (self._scalar("B") + 1, self._scalar("d")))
        if name in ("Pr_b", "theta"):
            return self._field(name, (self._scalar("B"),))
        if name == "sigma":
            return self._field(name, (self._scalar("K"),))
        if name == "lambda_":
            return self._field("lambda", (self._scalar("B") + 1,))
        if name == "B_vec":
            out = np.empty(self._scalar("C"), dtype=np.int32)
            self._L.hb_get_B_vec(self._h, _ptr(out))
            return out
        if name in TRACE:
            n = self._L.hb_trace(self._h, TRACE[name], None, 0)
            if n < 0:
                raise HarmonyError(self._L.hb_last_error(self._h).decode())
            out = np.empty(int(n), dtype=np.float64)
            self._L.hb_trace(self._h, TRACE[name], _ptr(out), n)
            return out.astype(np.int64) if name == "kmeans_rounds" else out
        raise AttributeError(name)

    def __setattr__(self, name, value):
        if name.startswith("_"):
            object.__setattr__(self, name, value)
            return
        if name in ("alpha", "max_iter_kmeans", "legacy_centroid_step", "kernel_set"):
            self._check(self._L.hb_set_scalar(self._h, SCALAR[name], float(value)))
            return
        shapes = {"Y": ("Y", "d", "K"), "R": ("R", "K", "N_local"), "O": ("O", "K", "B"), "E": ("E", "K", "B")}
        if name in shapes:
            f, r, c = shapes[name]
            v = np.asfortranarray(np.asarray(value, dtype=np.float64))
            if v.shape != (self._scalar(r), self._scalar(c)):
                raise ValueError(f"{name} must be {r} x {c}")
            self._check(self._L.hb_set_field(self._h, FIELD[f], _ptr(v)))
            return
        if name in ("theta", "sigma", "lambda_"):
            v = np.ascontiguousarray(value, dtype=np.float64)
            self._check(self._L.hb_set_field(self._h, FIELD["lambda" if name == "lambda_" else name], _ptr(v)))
            return
        raise AttributeError(f"field {name} is not writable")

    # ---- instrumentation -----------------------------------------------------------------------
    def synchronize(self):
        self._check(self._L.hb_synchronize(self._h))

    @property
    def kernel_launches(self):
        return int(self._L.hb_kernel_launches(self._h))

    @property
    def cuda_stream(self):
        return int(self._L.hb_stream(self._h) or 0)

    def enable_timing(self, on=True):
        self._L.hb_enable_timing(self._h, int(bool(on)))

    def region_time(self, region):
        ms, n = ctypes.c_double(), ctypes.c_int64()
        if self._L.hb_region_time(self._h, region.encode(), ctypes.byref(ms), ctypes.byref(n)) != 0:
            return 0.0, 0
        return ms.value, int(n.value)
