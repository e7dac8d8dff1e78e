"""Device-memory inputs and outputs (gpu-marked): hb_setup_device from CUDA tensors leaves the object in exactly the
state hb_setup leaves it in for the same values, to_torch returns exactly what the host getters return (as float32 /
float64), the caller's CUDA stream orders both, and full runs agree with the host-buffer runs."""
import os
import socket

import numpy as np
import pytest

from helpers import make_perms, make_Y0, rel_l2, synthetic

pytestmark = pytest.mark.gpu


def _torch():
    return pytest.importorskip("torch")


def _args(a):
    return (a["sigma"], a["theta"], a["lambda_"], a["alpha"], a["max_iter_kmeans"], a["epsilon_kmeans"],
            a["epsilon_harmony"], a["K"], a["block_size"], a["B_vec"], a["batch_proportion_cutoff"])


def _inputs(case):
    from harmony_b200 import prepare_inputs
    if case == "1cov":
        Z, meta = synthetic(20011, 30, [20], n_types=12, seed=31)
        return Z, prepare_inputs(Z, meta, "cov0", nclust=40, early_stop=False)
    if case == "3cov":
        Z, meta = synthetic(15013, 24, [4, 12, 3], seed=32)
        return Z, prepare_inputs(Z, meta, ["cov0", "cov1", "cov2"], nclust=30, early_stop=False)
    # key space 200^3 > 2^22: the dictionary falls back to the host implementation
    Z, meta = synthetic(6007, 16, [200, 200, 200], seed=33, nested=False)
    a = prepare_inputs(Z, meta, ["cov0", "cov1", "cov2"], nclust=20, early_stop=False)
    assert np.prod(a["B_vec"].astype(np.float64)) > 2 ** 22
    return Z, a


def _state(g):
    return dict(Z_orig=g.getZorig(), Z_corr=g.getZcorr(), Pr_b=g.Pr_b, B_vec=g.B_vec, perm=g.debug_sort_perm())


def _assert_same_state(x, y):
    for k in x:
        assert np.array_equal(x[k], y[k]), k


def _layouts(torch, Zd):
    """[N, d] contiguous, a [d, N] tensor's transpose view, and a column slice of a wider tensor."""
    N, d = Zd.shape
    wide = torch.zeros((N, d + 5), dtype=Zd.dtype, device=Zd.device)
    wide[:, 2:2 + d] = Zd
    return {"rows": Zd.contiguous(), "T_view": Zd.T.contiguous().T, "col_slice": wide[:, 2:2 + d]}


@pytest.mark.parametrize("case", ["1cov", "3cov", "big_key_space"])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_setup_state_identical(case, dtype):
    torch = _torch()
    from harmony_b200.harmony import harmony
    Z, a = _inputs(case)
    Zh = a["Z"].astype(dtype).astype(np.float64)           # the values both paths see
    h = harmony(device=0)
    h.setup(Zh, a["phi_i"], *_args(a))
    want = _state(h)
    Zd = torch.from_numpy(Zh).to(dtype=getattr(torch, dtype), device="cuda:0")
    for i, (name, Zt) in enumerate(_layouts(torch, Zd).items()):
        phi = a["phi_i"] if i % 2 == 0 else torch.from_numpy(a["phi_i"]).cuda()
        g = harmony(device=0)
        g.setup(Zt, phi, *_args(a))
        got = _state(g)
        for k in want:
            assert np.array_equal(got[k], want[k]), (name, k)


def test_outputs_identical():
    torch = _torch()
    from harmony_b200.harmony import harmony
    Z, a = _inputs("3cov")
    Y0 = make_Y0(Z, a["K"], 3)
    perms = make_perms(Z.shape[0], a["max_iter_kmeans"], 4)
    g = harmony(device=0)
    g.setup(torch.from_numpy(a["Z"]).cuda(), a["phi_i"], *_args(a))
    g.init_cluster_cpp(Y0)
    assert g.cluster_cpp(perms) == 0
    zc = g.to_torch("Z_corr")                              # applies the pending normalisation of cluster_cpp
    zc64 = g.to_torch("Z_corr", dtype=torch.float64)
    assert zc.dtype == torch.float32 and tuple(zc.shape) == (Z.shape[0], Z.shape[1])
    host = g.getZcorr().T
    assert np.array_equal(zc.cpu().numpy(), host.astype(np.float32))
    assert np.array_equal(zc64.cpu().numpy(), host)
    g.moe_correct_ridge_cpp()
    for f, get in (("Z_corr", g.getZcorr), ("Z_orig", g.getZorig), ("R", g.getR)):
        t = g.to_torch(f)
        assert np.array_equal(t.cpu().numpy(), get().T.astype(np.float32)), f
    d = Z.shape[1]
    wide = torch.full((Z.shape[0], d + 7), -1.0, dtype=torch.float64, device="cuda:0")
    out = g.to_torch("Z_corr", out=wide[:, 3:3 + d])
    assert out.data_ptr() == wide[:, 3:3 + d].data_ptr()
    assert np.array_equal(wide[:, 3:3 + d].cpu().numpy(), g.getZcorr().T)
    assert bool((wide[:, :3] == -1).all()) and bool((wide[:, 3 + d:] == -1).all())


def test_caller_stream_orders_inputs_and_outputs():
    torch = _torch()
    from harmony_b200.harmony import harmony
    Z, a = _inputs("1cov")
    h = harmony(device=0)
    h.setup(a["Z"], a["phi_i"], *_args(a))
    want = _state(h)
    src = torch.from_numpy(a["Z"]).cuda()
    phi_src = torch.from_numpy(a["phi_i"]).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = harmony(device=0)
    with torch.cuda.stream(side):
        torch.cuda._sleep(20_000_000)                      # Z and phi are written well after setup is called
        Zs = src * 1.0
        phi = phi_src + 0
        g.setup(Zs, phi, *_args(a))                        # no synchronise in between
    _assert_same_state(_state(g), want)
    out = g.to_torch("Z_orig") * 1.0                       # consumed on the current stream, no synchronise
    assert np.array_equal(out.cpu().numpy(), want["Z_orig"].T.astype(np.float32))


def test_full_run_matches_host_path():
    torch = _torch()
    from harmony_b200.harmony import harmony
    Z, a = _inputs("3cov")
    Y0 = make_Y0(Z, a["K"], 5)
    T = a["max_iter_kmeans"]
    perms = make_perms(Z.shape[0], 2 * T, 6).reshape(2, T, -1)
    res = []
    for Zin in (a["Z"], torch.from_numpy(a["Z"]).cuda()):
        g = harmony(device=0)
        g.setup(Zin, a["phi_i"], *_args(a))
        g.init_cluster_cpp(Y0)
        for it in range(2):
            assert g.cluster_cpp(perms[it]) == 0
            g.moe_correct_ridge_cpp()
            g.check_convergence(1)
        res.append(g.getZcorr())
    assert rel_l2(res[1], res[0]) < 1e-5


@pytest.mark.parametrize("dtype, tensor_meta", [("float64", False), ("float32", False), ("float32", True)])
def test_runharmony_on_cuda_tensor(dtype, tensor_meta):
    torch = _torch()
    from harmony_b200 import RunHarmony
    Z, meta = synthetic(5000, 20, [4], seed=9)
    Z = Z.astype(dtype)
    want = RunHarmony(Z.astype(np.float64), meta, "cov0", nclust=20, max_iter=3, verbose=False, seed=11)
    Zt = torch.from_numpy(Z).cuda()
    m = {"cov0": torch.from_numpy(meta["cov0"]).cuda()} if tensor_meta else meta
    got = RunHarmony(Zt.T, m, "cov0", nclust=20, max_iter=3, verbose=False, seed=11)   # [d, N] given: transposed
    assert got.is_cuda and got.dtype == Zt.dtype and tuple(got.shape) == Z.shape
    assert rel_l2(got.double().cpu().numpy(), want) < 1e-5
    obj = RunHarmony(Zt, m, "cov0", nclust=20, max_iter=1, verbose=False, seed=11, return_object=True)
    assert obj.getZcorr().shape == (Z.shape[1], Z.shape[0])


def test_errors_match_host_path():
    torch = _torch()
    from harmony_b200.harmony import HarmonyError, harmony
    Z, a = _inputs("3cov")
    phi = a["phi_i"].copy()
    phi[4567, 1] = 3          # a level of covariate 0 given for covariate 1 ...
    phi[123, 2] = 99          # ... and a row past every level: the host path reports the lower cell
    with pytest.raises(HarmonyError) as host_err:
        harmony(device=0).setup(a["Z"], phi, *_args(a))
    assert "cell 123 " in str(host_err.value)
    with pytest.raises(HarmonyError) as dev_err:
        harmony(device=0).setup(torch.from_numpy(a["Z"]).cuda(), torch.from_numpy(phi).cuda(), *_args(a))
    assert str(dev_err.value) == str(host_err.value)
    with pytest.raises(TypeError, match="float32 or float64"):
        harmony(device=0).setup(torch.from_numpy(a["Z"]).half().cuda(), a["phi_i"], *_args(a))
    with pytest.raises(ValueError, match="2-D"):
        harmony(device=0).setup(torch.from_numpy(a["Z"]).cuda()[None], a["phi_i"], *_args(a))
    g = harmony(device=0)                                  # host memory where device memory is due (C ABI)
    L = g._L
    Zh = np.ascontiguousarray(a["Z"])
    phi_d = torch.from_numpy(a["phi_i"]).cuda()
    B_vec, sigma, theta = a["B_vec"], np.ascontiguousarray(a["sigma"]), np.ascontiguousarray(a["theta"])
    st = L.hb_setup_device(g._h, Zh.ctypes.data, 1, Zh.shape[1], 1, Zh.shape[1], Zh.shape[0], phi_d.data_ptr(),
                           B_vec.ctypes.data, len(B_vec), sigma.ctypes.data, theta.ctypes.data, None, 0.2,
                           a["max_iter_kmeans"], 1e-3, -np.inf, a["K"], 0.05, 1e-5, 0, None)
    assert st != 0 and "Z is not CUDA device memory" in L.hb_last_error(g._h).decode()
    with pytest.raises(ValueError, match="field"):
        h = harmony(device=0)
        h.setup(torch.from_numpy(a["Z"]).cuda(), a["phi_i"], *_args(a))
        h.to_torch("Y")
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="cuda:1"):
            harmony(device=0).setup(torch.from_numpy(a["Z"]).to("cuda:1"), a["phi_i"], *_args(a))


# ---- two GPUs: sharded hb_setup_device == sharded hb_setup, rank by rank --------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run_sharded(rank, world, port, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import torch
    import torch.distributed as dist
    from harmony_b200 import prepare_inputs
    from harmony_b200.dist import make_comm, shard_bounds
    from harmony_b200.harmony import harmony
    from helpers import synthetic as synth
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        Z, meta = synth(20007, 24, [4, 12, 3], seed=12)
        a = prepare_inputs(Z, meta, ["cov0", "cov1", "cov2"], nclust=40, early_stop=False)
        N = Z.shape[0]
        lo, hi = shard_bounds(N, world, rank)
        args = (a["sigma"], a["theta"], a["lambda_"], a["alpha"], a["max_iter_kmeans"], a["epsilon_kmeans"],
                a["epsilon_harmony"], a["K"], a["block_size"], a["B_vec"], a["batch_proportion_cutoff"])
        comm = make_comm(N)
        gh = harmony(device=rank, comm=comm)
        gh.setup(a["Z"][lo:hi], a["phi_i"][lo:hi], *args)
        gd = harmony(device=rank, comm=(comm[0], comm[1], None, comm[3], comm[4]))
        gd.setup(torch.from_numpy(a["Z"][lo:hi]).cuda(rank), torch.from_numpy(a["phi_i"][lo:hi]).cuda(rank), *args)
        same = {}
        for k, f in (("perm", lambda g: g.debug_sort_perm()), ("Pr_b", lambda g: g.Pr_b), ("Z_orig", lambda g: g.getZorig()),
                     ("N_local", lambda g: g._scalar("N_local"))):
            same[k] = bool(np.array_equal(f(gh), f(gd)))
        dist.barrier()
        q.put((rank, same))
    except Exception:  # pragma: no cover
        import traceback
        q.put((rank, "ERR " + traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def test_two_gpu_sharded_setup_identical():
    torch = _torch()
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_run_sharded, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for r, v in res.items():
        assert not isinstance(v, str), v
        assert all(v.values()), (r, v)
