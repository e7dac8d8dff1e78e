"""``RunHarmony`` — host-side mirror of /root/reference/R/ui.R:91-309 (``RunHarmony.default``).

Only argument preparation lives here (the reference does it in R too); all arithmetic on the
cell matrices happens behind the C ABI (include/harmony_b200.h) in hand-written CUDA.
"""
import math
import os
import sys

import numpy as np

from .harmony import torch_of
from .harmony_option import HarmonyOptions, check_legacy_args, harmony_options
from .utils import harmonize


def _column(v):
    """A covariate column as a 1-D array; CUDA tensors stay on their device."""
    torch = torch_of(v)
    return v if torch is not None and v.is_cuda else np.asarray(v)


def _as_columns(meta_data, n_hint):
    """meta_data -> dict name -> 1-D array (or CUDA tensor).  Accepts a dict, a pandas DataFrame or one vector
    (R/ui.R:157-165: a bare vector becomes data.frame(batch_variable = ...))."""
    if hasattr(meta_data, "columns") and hasattr(meta_data, "__getitem__") and not isinstance(meta_data, dict):
        return {str(c): np.asarray(meta_data[c]) for c in meta_data.columns}, None
    if isinstance(meta_data, dict):
        return {str(k): _column(v) for k, v in meta_data.items()}, None
    v = _column(meta_data)
    if v.ndim == 1 and len(v) in n_hint:
        return {"batch_variable": v}, "batch_variable"
    raise ValueError("meta_data must be either a data.frame or a vector with batch values for each cell")


def prepare_inputs(data_mat, meta_data, vars_use=None, theta=None, sigma=0.1, lambda_=None, nclust=None,
                   early_stop=True, options=None, verbose=False):
    """Everything RunHarmony.default computes before ``new(harmony)`` (R/ui.R:133-258).

    Returns a dict with the exact argument list of ``harmony::setup`` (src/harmony.h:25-30), with
    the sparse ``phi`` expressed as its row-index slot: ``phi_i[n, c]`` = row of the c-th non-zero of
    column n (each cell has exactly one level per covariate, so columns hold C non-zeros).

    A CUDA tensor ``data_mat`` stays on its device: ``Z`` is that tensor (or its transpose view) and ``phi_i`` an int32
    tensor on the same device.  Covariate columns may be CUDA integer tensors; their levels are
    ``torch.unique(sorted=True)``, the order ``np.unique`` gives.
    """
    options = harmony_options() if options is None else options
    if not isinstance(options, HarmonyOptions):
        raise TypeError("Error: .options must be created from harmony_options()!")
    epsilon_harmony = options.epsilon_harmony if early_stop else -math.inf
    torch = torch_of(data_mat)
    on_device = torch is not None and data_mat.is_cuda
    if not on_device:
        data_mat = np.asarray(data_mat)
    if data_mat.ndim != 2:
        raise ValueError("data_mat must be a matrix")
    cols, forced = _as_columns(meta_data, data_mat.shape)
    if forced is not None:
        vars_use = forced
    if vars_use is None:
        raise ValueError("must provide variables names (e.g. vars_use='stim')")
    if isinstance(vars_use, str):
        vars_use = [vars_use]
    vars_use = list(vars_use)
    if any(v not in cols for v in vars_use):
        raise ValueError("must provide variables names (e.g. vars_use='stim')")
    N = len(next(iter(cols.values())))
    # R/ui.R:178-189: cells must end up as columns; here the row-major [N, d] view is the same bytes
    if data_mat.shape[0] == N:
        Z = data_mat
    elif data_mat.shape[1] == N:
        if verbose:
            print("Transposing data matrix", file=sys.stderr)
        Z = data_mat.T
    else:
        raise ValueError("number of labels do not correspond to number of samples in data matrix")
    if nclust is None:
        nclust = min(int(round(N / 30.0)), 100)
    if theta is None:
        theta = [2.0] * len(vars_use)
    else:
        theta = list(np.atleast_1d(np.asarray(theta, dtype=np.float64)))
        if len(theta) != len(vars_use):
            raise ValueError("Please specify theta for each variable")
    sigma = np.atleast_1d(np.asarray(sigma, dtype=np.float64))
    if len(sigma) == 1 and nclust > 1:
        sigma = np.repeat(sigma, nclust)
    # phi / B_vec: as.factor levels = sorted unique values (R/ui.R:210-221)
    phi_cols, B_vec, level_names = [], [], []
    offset = 0
    for v in vars_use:
        col, tc = cols[v], torch_of(cols[v])
        if tc is not None:                                            # a CUDA tensor column
            levels, codes = tc.unique(col, sorted=True, return_inverse=True)
            codes = codes.to(tc.int32) + offset
            if not on_device:
                codes = codes.cpu().numpy()
            levels = levels.cpu().numpy()
        else:
            levels, codes = np.unique(col, return_inverse=True)
            codes = codes.astype(np.int32) + offset
            if on_device:
                codes = torch.from_numpy(codes).to(data_mat.device)
        phi_cols.append(codes)
        B_vec.append(len(levels))
        level_names.append(levels)
        offset += len(levels)
    B = offset
    if on_device:
        phi_i = torch.stack(phi_cols, dim=1).contiguous()             # [N, C] on the device
        N_b = torch.bincount(phi_i.reshape(-1).long(), minlength=B).cpu().numpy().astype(np.float64)
    else:
        phi_i = np.ascontiguousarray(np.stack(phi_cols, axis=1))      # [N, C]
        N_b = np.bincount(phi_i.reshape(-1), minlength=B).astype(np.float64)
    if lambda_ is None:                                               # R/ui.R:224-229
        lambda_vec = None
    else:
        lam = np.atleast_1d(np.asarray(lambda_, dtype=np.float64))
        if not np.all(lam > 0):
            raise ValueError("Provided lambdas must be positive")
        if len(lam) == 1:
            lambda_vec = np.concatenate([[0.0], np.repeat(lam, B)])
        else:
            if len(lam) != len(vars_use):
                raise ValueError(
                    f"You specified a lambda value for each covariate but the number of lambdas specified "
                    f"({len(lam)}) and the number of covariates ({len(vars_use)}) mismatch.")
            lambda_vec = np.concatenate([[0.0], np.repeat(lam, B_vec)])
    theta_vec = np.repeat(np.asarray(theta, dtype=np.float64), B_vec)
    tau = options.tau
    with np.errstate(divide="ignore", invalid="ignore"):              # tau = 0 -> N_b/0 = Inf -> factor 1
        theta_vec = theta_vec * (1 - np.exp(-(N_b / (nclust * tau)) ** 2)) if tau != 0 else theta_vec * 1.0
    return dict(Z=Z if on_device else np.ascontiguousarray(Z, dtype=np.float64), phi_i=phi_i, B_vec=np.asarray(B_vec, dtype=np.int32),
                sigma=sigma, theta=theta_vec, lambda_=lambda_vec, alpha=float(options.alpha),
                max_iter_kmeans=int(options.max_iter_cluster), epsilon_kmeans=float(options.epsilon_cluster),
                epsilon_harmony=float(epsilon_harmony), K=int(nclust), block_size=float(options.block_size),
                batch_proportion_cutoff=float(options.batch_prop_cutoff), level_names=level_names,
                vars_use=vars_use)


def RunHarmony(data_mat, meta_data, vars_use=None, theta=None, sigma=0.1, lambda_=None, nclust=None, max_iter=10,
               early_stop=True, ncores=1, plot_convergence=False, return_object=False, verbose=True,
               options=None, seed=None, device=None, **kwargs):
    """RunHarmony.default (R/ui.R:91-309) on B200.

    ``ncores`` (CPU BLAS threads, R/ui.R:101,123-128) is accepted and ignored; ``seed`` replaces R's
    ``set.seed`` for the k-means initialisation and the per-round update orders.  Returns the
    corrected embedding [N, d] (same orientation rule as the reference: the transpose of what
    ``getZcorr()`` holds) or the ``harmony`` object when ``return_object`` is true.

    A CUDA tensor ``data_mat`` runs on its device without host copies of the cell data and returns a CUDA tensor
    [N, d] of its dtype (see ``prepare_inputs`` for covariate columns held as CUDA tensors).
    """
    from .harmony import harmony  # needs the CUDA extension; fails loudly when it is missing

    check_legacy_args(**kwargs)
    a = prepare_inputs(data_mat, meta_data, vars_use, theta, sigma, lambda_, nclust, early_stop, options, verbose)
    if verbose and a["lambda_"] is None:
        print("Using automatic lambda estimation", file=sys.stderr)
    torch = torch_of(a["Z"])
    if torch is not None and device is None:
        device = a["Z"].device.index
    obj = harmony(device=device)
    obj.setup(a["Z"], a["phi_i"], a["sigma"], a["theta"], a["lambda_"], a["alpha"], a["max_iter_kmeans"],
              a["epsilon_kmeans"], a["epsilon_harmony"], a["K"], a["block_size"], a["B_vec"],
              a["batch_proportion_cutoff"], verbose)
    if seed is None:   # R without set.seed(): the session's random stream differs from run to run
        seed = int.from_bytes(os.urandom(8), "little")
    obj.set_seed(seed)
    if verbose:
        print("Initializing state using k-means centroids initialization", file=sys.stderr)
    obj.init_cluster_cpp()
    harmonize(obj, max_iter, verbose)
    if plot_convergence:
        from .utils import HarmonyConvergencePlot
        HarmonyConvergencePlot(obj)
    if return_object:
        return obj
    if torch is not None:
        return obj.to_torch("Z_corr", dtype=a["Z"].dtype)
    return np.ascontiguousarray(obj.getZcorr().T)   # t(harmonyObj$getZcorr()), R/ui.R:292-295: cells x PCs
