#!/usr/bin/env python
"""bench.py — cells / second / Harmony-iteration on synthetic embeddings (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One *step* = one trip of the harmonize() loop body (R/utils.R:20-45): cluster_cpp (cold-start
re-estimate + T=4 x (update_R + compute_objective)) + moe_correct_ridge_cpp + check_convergence(1),
defaults of R/harmony_option.R:33-40, early_stop = FALSE.  Workload at N=1: BASELINE.json config 3
(synthetic 1M cells x 50 PCs, 1 covariate with 20 batches, K=100).  Weak scaling: every rank holds
CELLS_PER_GPU cells of one global problem (cells sharded, global statistics all-reduced).

The JSON line carries `value` (device-resident, CUDA-event timed on the library's stream, max over
ranks), `e2e` (the same metric through the public API with HOST buffers: setup H2D + init + iterations +
getZcorr D2H), `roofline` (dominant kernel, algorithmic bytes / measured launch time, against
MEASURED_PEAKS.json) and `cpu_baseline` (the CPU oracle = restatement of the reference, timed on this
box's host cores on a bounded sample).

`--dump-outputs DIR` writes what the timed path handed its caller after the last timed step (see dump_outputs), so
that two builds run with the same arguments, and therefore the same inputs, can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T = 4
N_TYPES = 30
# BASELINE.json configs 3 / 4 / 5 as PER-GPU shards (config 4: 10M cells over 8 GPUs, config 5: 50M over 8);
# the headline metric is quoted on config 3.  Level counts beyond config 3's are SURVEY.md 8(d)'s stated choice.
WORKLOADS = {
    "c3": dict(cells_per_gpu=1_000_000, d=50, K=100, B_vec=[20],
               name="BASELINE.json config 3 per GPU", metric="cells/sec/Harmony-iteration (50 PCs, K=100)"),
    "c4": dict(cells_per_gpu=1_250_000, d=50, K=100, B_vec=[10, 40],
               name="BASELINE.json config 4 (10M cells, dataset + donor) as the per-GPU shard of 8",
               metric="cells/sec/Harmony-iteration (50 PCs, K=100, 2 covariates)"),
    "c5": dict(cells_per_gpu=6_250_000, d=100, K=200, B_vec=[10, 40, 6],
               name="BASELINE.json config 5 (50M cells, 3 covariates) as the per-GPU shard of 8",
               metric="cells/sec/Harmony-iteration (100 PCs, K=200, 3 covariates)"),
}
W = dict(WORKLOADS["c3"])   # the active workload (set in main)


def algo_bytes_per_cell_iter(K, d):
    """SURVEY.md 8(d): algorithmic bytes per cell per Harmony iteration, fp32 state, T rounds."""
    return 4 * (K * (3 + 2 * T) + d * (5 + T)) + 4 * (T + 2)   # 6224 for K=100, d=50; 12424 for K=200, d=100


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def synth_shard(n, cell_offset, seed, d=None, B_vec=None, n_types=N_TYPES):
    """SURVEY.md 8(d) generator: Z[i,j] = sd_j (M[t_i,j] + sum_c 0.5 S_c[b_ci,j] + 0.6 eps), sd_j = 10/sqrt(1+j);
    type probabilities ~ Dirichlet(2), level probabilities ~ LogNormal(0, 0.5).  Further covariates are NESTED:
    every level of covariate c >= 1 ("donor") belongs to one level of covariate 0 ("dataset", levels dealt round
    robin), a third covariate is a fixed property of the donor -> J = #donors joint tuples.  Global parameters
    come from `seed`, the per-cell draws from (seed, cell_offset) so shards are consistent for any world size.
    Returns Z (float64, n x d) and the level ids (int32, n x C, per-covariate numbering)."""
    d = W["d"] if d is None else d
    B_vec = W["B_vec"] if B_vec is None else B_vec
    g = np.random.default_rng(seed)
    M = g.standard_normal((n_types, d)).astype(np.float32)
    S = [g.standard_normal((b, d)).astype(np.float32) for b in B_vec]
    p_type = g.dirichlet(np.full(n_types, 2.0))
    p_lvl = [g.lognormal(0.0, 0.5, b) for b in B_vec]
    chem_of_donor = g.integers(0, B_vec[2], B_vec[1]) if len(B_vec) > 2 else None
    sd = (10.0 / np.sqrt(1.0 + np.arange(d))).astype(np.float32)
    r = np.random.default_rng([seed, cell_offset])
    t = r.choice(n_types, n, p=p_type)
    lv = np.empty((n, len(B_vec)), dtype=np.int32)
    lv[:, 0] = r.choice(B_vec[0], n, p=p_lvl[0] / p_lvl[0].sum())
    if len(B_vec) > 1:
        parent = np.arange(B_vec[1]) % B_vec[0]
        for p in range(B_vec[0]):
            cand = np.flatnonzero(parent == p)
            sel = np.flatnonzero(lv[:, 0] == p)
            w = p_lvl[1][cand]
            lv[sel, 1] = r.choice(cand, sel.size, p=w / w.sum())
    if len(B_vec) > 2:
        lv[:, 2] = chem_of_donor[lv[:, 1]]
    Z = M[t] + 0.6 * r.standard_normal((n, d), dtype=np.float32)
    for c in range(len(B_vec)):
        Z += 0.5 * S[c][lv[:, c]]
    Z *= sd[None, :]
    return Z.astype(np.float64), lv


def host_Y0(Z, k, seed):
    """Initial centroids (stand-in for kmeans_centers, outside the timed path): k distinct random cells of
    a subsample + 2 Lloyd iterations on the cosine-normalised subsample."""
    rng = np.random.default_rng(seed)
    sub = Z[rng.choice(Z.shape[0], min(Z.shape[0], 50_000), replace=False)]
    sub = sub / np.maximum(np.linalg.norm(sub, axis=1, keepdims=True), 1e-30)
    Y = sub[rng.choice(sub.shape[0], k, replace=False)].copy()
    for _ in range(2):
        a = np.argmax(sub @ Y.T, axis=1)
        for j in range(k):
            if np.any(a == j):
                Y[j] = sub[a == j].mean(axis=0)
    return Y


def setup_kwargs(lv):
    """Defaults of R/ui.R:95-100 / R/harmony_option.R:33-40; level ids renumbered globally (covariate c's levels
    follow those of covariate c - 1), as R/ui.R:219-231 builds Phi."""
    B_vec = np.asarray(W["B_vec"], dtype=np.int32)
    off = np.concatenate([[0], np.cumsum(B_vec)[:-1]]).astype(np.int32)
    return dict(phi=np.ascontiguousarray(lv + off[None, :]), sigma=np.full(W["K"], 0.1), theta=np.full(int(B_vec.sum()), 2.0),
                lambda_=None, alpha=0.2, max_iter_kmeans=T, epsilon_kmeans=1e-3, epsilon_harmony=-np.inf, K=W["K"],
                block_size=0.05, B_vec=B_vec, cutoff=1e-5)


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region (B200_PROFILING.md recipe).  NVML is polled every
    few milliseconds (the timed region lasts tens of ms); nvidia-smi is the fallback."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, period=0.003):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self._halt, self.period = gpu_index, [], threading.Event(), period
        self.nvml = None
        self.marked = 0
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = gpu_index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                idx = int(vis.split(",")[gpu_index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll_nvml(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        self.rows.append((sm, self.max_sm, mask))

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                if self.nvml is not None:
                    self._poll_nvml()
                    self._halt.wait(self.period)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    r = [x.strip() for x in out.stdout.strip().split(",")]
                    mask = 0
                    for bit, col in ((0x8, 3), (0x40, 4), (0x20, 5), (0x4, 6)):
                        if len(r) > col and r[col].lower().startswith("active"):
                            mask |= bit
                    self.rows.append((float(r[0]), float(r[1]), mask))
            except Exception:
                pass
            self._halt.wait(0.2)

    def mark(self):
        """Samples taken from now on fall into the timed region."""
        self.marked = len(self.rows)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows]
        mask = 0
        for r in self.rows:
            mask |= r[2]
        reasons = [nm for bit, nm in self.REASONS.items() if mask & bit]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows), "samples_in_timed_region": len(self.rows) - self.marked,
                "how": "dense sampling over 5 untimed steps of the same loop right before the timed region, sparse inside it",
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def measured_traffic(kernel, config, n_local):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernel from the committed
    ncu --set full capture of this workload (profiles/traffic.json: {config: {kernel: {"cells": n, "bytes": b}}});
    None when no capture of this kernel at this shard size has been committed."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[config][kernel]
        return float(t["bytes"]) if int(t["cells"]) == int(n_local) else None
    except Exception:
        return None


def cpu_sample_cells():
    """Bounded CPU sample: ~200k cells at K=100, d=50 (about 5 s per oracle iteration), fewer for wider shapes."""
    return int(max(20_000, min(200_000, 200_000 * (100 * 50) / (W["K"] * W["d"]))))


def cpu_reference_run(n_cells, iters, threads, seed=20260925, keep=None):
    """Times the CPU oracle (restatement of the reference's Armadillo/OpenBLAS path) on host cores.  `keep` (a dict)
    receives the inputs and the oracle's final state so that the caller can hold the GPU path against them."""
    from oracle.oracle import OracleHarmony, load_blas
    blas = load_blas(threads)
    Z, b = synth_shard(n_cells, 0, seed)
    kw = setup_kwargs(b)
    K = W["K"]
    Y0 = host_Y0(Z, K, 1)
    o = OracleHarmony()
    o.setup(Z, kw["phi"], kw["B_vec"], kw["sigma"], kw["theta"], None, kw["alpha"], T, 1e-3, -np.inf, K, 0.05, 1e-5)
    o.init_cluster_cpp(Y0)
    rng = np.random.default_rng(5)
    times, all_perms = [], []
    for it in range(iters + 1):             # iteration 1 skips the cold start -> untimed
        perms = np.stack([rng.permutation(n_cells) for _ in range(T)]).astype(np.int64)
        all_perms.append(perms)
        t0 = time.perf_counter()
        o.cluster_cpp(perms)
        o.moe_correct_ridge_cpp()
        o.check_convergence(1)
        if it > 0:
            times.append(time.perf_counter() - t0)
    if keep is not None:
        keep.update(Z=Z, kw=kw, Y0=Y0, perms=all_perms, Z_corr=o.get("Z_corr"), R=o.get("R"))
    return float(np.median(times)), blas


def parity_on_sample(device, n_cells=50_000, iters=2, seed=20260926):
    """The GPU path against the CPU oracle (the checker) on a bounded sample of the workload, same centroids and update
    orders: rel-L2 of the corrected embedding against the reference-order fp32 oracle AND against its fp64 instance
    (the fp32 oracle's own sequential-sum noise grows with N: tests/test_gpu_parity.py), and the number of cells
    whose hard cluster index differs."""
    from harmony_b200.harmony import harmony
    from oracle.oracle import OracleHarmony
    Z, b = synth_shard(n_cells, 0, seed)
    kw = setup_kwargs(b)
    K = W["K"]
    Y0 = host_Y0(Z, K, 1)
    rng = np.random.default_rng(7)
    perms = [np.stack([rng.permutation(n_cells) for _ in range(T)]).astype(np.int64) for _ in range(iters)]
    res = {}
    for name, dbl in (("oracle32", False), ("oracle64", True)):
        o = OracleHarmony(double=dbl)
        o.setup(Z, kw["phi"], kw["B_vec"], kw["sigma"], kw["theta"], None, kw["alpha"], T, 1e-3, -np.inf, K, 0.05, 1e-5)
        o.init_cluster_cpp(Y0)
        for p in perms:
            o.cluster_cpp(p)
            o.moe_correct_ridge_cpp()
            o.check_convergence(1)
        res[name] = (o.get("Z_corr"), o.get("R"))
    g = harmony(device=device)
    g.setup(Z, kw["phi"], kw["sigma"], kw["theta"], None, kw["alpha"], T, 1e-3, -np.inf, K, 0.05, kw["B_vec"], kw["cutoff"])
    g.init_cluster_cpp(Y0)
    for p in perms:
        assert g.cluster_cpp(p) == 0
        g.moe_correct_ridge_cpp()
        g.check_convergence(1)
    Zg, Rg = g.getZcorr().T, g.R.T
    out = {"cells": int(n_cells), "iterations": iters}
    for name, (Zo, Ro) in res.items():
        part = np.partition(Ro, -2, axis=1)
        gap = part[:, -1] - part[:, -2]
        diff = Rg.argmax(axis=1) != Ro.argmax(axis=1)
        out[name] = {"rel_l2_Z": float(np.linalg.norm(Zg - Zo) / np.linalg.norm(Zo)), "argmax_mismatch": int(diff.sum()),
                     "largest_oracle_top2_gap_among_them": float(gap[diff].max()) if diff.any() else 0.0,
                     "max_abs_dR": float(np.abs(Rg - Ro).max())}
    Z32, Z64 = res["oracle32"][0], res["oracle64"][0]
    out["oracle32_vs_oracle64_rel_l2_Z"] = float(np.linalg.norm(Z32 - Z64) / np.linalg.norm(Z64))
    return out


DUMP_CELLS = 32_768     # 39 MB of float32 at the widest workload (c5: d=100, K=200)


def dump_outputs(g, n_local, out_dir, seed=20261017):
    """Writes DIR/<name>.npy: the corrected embedding (getZcorr, d x cells) and the soft cluster assignments
    (R, K x cells) of a fixed, seeded sample of DUMP_CELLS cells of this rank's shard, in shard order, the
    centroids (Y, d x K) and the last Harmony objective.  The library holds its state in fp32, so Z_corr, R and Y
    are stored as float32 without loss; the objective stays float64."""
    os.makedirs(out_dir, exist_ok=True)
    cells = np.sort(np.random.default_rng(seed).choice(n_local, min(n_local, DUMP_CELLS), replace=False))
    out = {"Z_corr": g.getZcorr()[:, cells].astype(np.float32),      # one full download at a time
           "R": g.getR()[:, cells].astype(np.float32),
           "Y": g.getCentroids().astype(np.float32),
           "objective_harmony": g.objective_harmony[-1:].astype(np.float64)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))
    log(f"outputs of the last timed step written to {out_dir}: "
        + ", ".join(f"{k} {v.shape} {v.dtype}" for k, v in out.items()))


def run_reference(args):
    """--impl reference: the reference's own CPU algorithm (oracle port) with all host BLAS threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncpu = os.cpu_count() or 1
    n_sample = int(args.ref_cells) if args.ref_cells > 0 else cpu_sample_cells()
    steps = args.steps
    # the reference only threads its BLAS call (R/ui.R:123-128); time it with all host threads and with the
    # reference default ncores = 1 and report the faster of the two (skinny sgemm often loses with threads)
    t_all, blas = cpu_reference_run(n_sample, steps, ncpu)
    t_one, _ = cpu_reference_run(n_sample, steps, 1) if ncpu > 1 else (t_all, blas)
    t_iter, cores = (t_all, ncpu) if t_all <= t_one else (t_one, 1)
    v = n_sample / t_iter
    D, K = W["d"], W["K"]
    line = {"impl": "reference", "metric": W["metric"], "value": v, "unit": "cells/s/iter", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": t_iter * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"synthetic {n_sample} cells x {D} PCs, {len(W['B_vec'])} covariate(s) (levels {W['B_vec']}), "
                                   f"K={K} (bounded sample of {W['name']}; the algorithm is O(N))"},
            "cpu_baseline": {"value": v, "unit": "cells/s/iter", "cores": cores, "kind": "port",
                             "sample": f"{n_sample} cells, {steps} timed iteration(s), BLAS={os.path.basename(blas)}; "
                                       f"all {ncpu} threads: {n_sample / t_all:.0f} cells/s/iter, 1 thread: "
                                       f"{n_sample / t_one:.0f} cells/s/iter (faster one reported)"},
            "e2e": {"value": v, "unit": "cells/s/iter", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(WORKLOADS), help="BASELINE.json workload (per-GPU shard)")
    ap.add_argument("--cells-per-gpu", type=int, default=0, help="override the workload's shard size")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--clock-period", type=float, default=0.003, help="seconds between NVML clock samples during the timed region")
    ap.add_argument("--kernel-set", type=int, default=0, help="HB_KERNEL_SET test hook of the library (A/B runs only)")
    ap.add_argument("--ref-cells", type=int, default=0, help="cells of the bounded CPU sample (--impl reference); 0 = by workload")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (rank 0's shard; --impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    W.clear()
    W.update(WORKLOADS[args.config])
    if args.cells_per_gpu <= 0:
        args.cells_per_gpu = W["cells_per_gpu"]
    D, K, METRIC = W["d"], W["K"], W["metric"]
    ALGO_BYTES_PER_CELL_ITER = algo_bytes_per_cell_iter(K, D)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from harmony_b200.harmony import harmony
    from harmony_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        log(f"warning: WORLD_SIZE={world} but --gpus {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    n_local = args.cells_per_gpu
    N_global = n_local * world
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    comm_made = []

    def new_comm():
        """First object: a fresh NCCL unique id (usable once); later objects share the process-wide
        communicator (id = None), as a long-lived service would."""
        if world == 1:
            return None
        if comm_made:
            return (rank, world, None, N_global, rank * n_local)
        comm_made.append(1)
        import ctypes
        uid = ctypes.create_string_buffer(128)
        if rank == 0:
            assert _lib.lib().hb_comm_unique_id(uid) == 0
        t = torch.tensor(list(uid.raw), dtype=torch.uint8, device="cuda")
        dist.broadcast(t, 0)
        return (rank, world, bytes(t.cpu().tolist()), N_global, rank * n_local)

    seed = 20260922 + int(args.config[1:])
    Z, b = synth_shard(n_local, rank * n_local, seed)
    kw = setup_kwargs(b)
    Y0 = host_Y0(Z, K, 1) if rank == 0 else np.zeros((K, D))
    if world > 1:
        ty = torch.from_numpy(Y0).cuda()
        dist.broadcast(ty, 0)
        Y0 = ty.cpu().numpy()

    def make_obj():
        g = harmony(device=local_rank, comm=new_comm())
        if args.kernel_set:
            g.kernel_set = args.kernel_set
        g.setup(Z, kw["phi"], kw["sigma"], kw["theta"], None, kw["alpha"], T, 1e-3, -np.inf, K, 0.05, kw["B_vec"],
                kw["cutoff"])
        g.set_seed(1234)
        g.init_cluster_cpp(Y0)
        return g

    def step(g):
        st = g.cluster_cpp()
        assert st == 0
        g.moe_correct_ridge_cpp()
        g.check_convergence(1)

    g = make_obj()
    stream = torch.cuda.ExternalStream(g.cuda_stream, device=torch.device("cuda", local_rank))
    for _ in range(max(3, args.warmup)):
        step(g)
    g.synchronize()
    # Clocks under load.  NVML queries perturb sharded runs badly (measured on 2 x B200: a query every 3 ms inside the
    # timed loop turns 2.9 ms per iteration into 5.0 — the ranks run in lockstep, every stall of one GPU is a stall of
    # all; a single GPU does not notice).  So the same steps run untimed once more under dense sampling (the load and
    # therefore the clocks are those of the timed region), and inside the timed region the sampler only looks a couple
    # of times (period = a third of the region's expected length).
    sampler = ClockSampler(local_rank, args.clock_period) if rank == 0 else None
    t_probe = time.perf_counter()
    if sampler:
        sampler.start()
    probe_steps = 5
    for _ in range(probe_steps):
        step(g)
    g.synchronize()
    t_probe = (time.perf_counter() - t_probe) / probe_steps
    if sampler:
        sampler.period = max(args.clock_period, min(0.5, t_probe * args.steps / 3.0))
        sampler.mark()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = g.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step(g)
    e1.record(stream)
    g.synchronize()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = g.kernel_launches - l0
    if world > 1:
        dist.barrier()
        tm = torch.tensor([ms], device="cuda")
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ms = float(tm.item())
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(g, n_local, args.dump_outputs)
    ms_per_step = ms / args.steps
    value = N_global / (ms_per_step * 1e-3)

    # ---- per-kernel timing pass (region timers: CUDA events on the library stream, extra syncs) -> roofline
    peaks, peak_kind = measured_peaks()
    g.enable_timing(True)
    names = ("k_update_steps", "k_rem_sums", "k_update_finalize", "k_block_update", "k_block_colsum", "k_step_prepare", "assign",
             "plan", "ridge_stats", "ridge_solve", "ridge_apply", "update_R")
    base = {r: g.region_time(r) for r in names}
    prof_steps = 3
    for _ in range(prof_steps):
        step(g)
    g.synchronize()
    reg = {}
    for r, (ms0, n0) in base.items():
        ms1, n1 = g.region_time(r)
        reg[r] = {"ms_per_step": (ms1 - ms0) / prof_steps, "launches_per_step": (n1 - n0) / prof_steps}
    g.enable_timing(False)
    KS, DS, nb = (K + 3) // 4 * 4, (D + 3) // 4 * 4, 20
    # algorithmic bytes per cell of each hot kernel (DESIGN.md section 3), fp32
    algo = {
        # all T rounds in one launch: per round the U row + its order / previous-block entries; R stored once
        "k_update_steps": T * (4 * KS + 8) + 4 * KS,
        "k_block_update": (8 * KS + 4) / nb,            # v1 fallback: one block per launch
        "assign": 8 * DS + 8 * KS,                       # Zc in/out, U and R out
        "ridge_stats": 4 * KS + 4 * DS,                  # R and Zo in
        "ridge_apply": 4 * KS + 8 * DS,                  # R and Zo in, Zc out
    }
    timed = {r: reg[r]["ms_per_step"] for r in ("k_update_steps", "k_block_update", "assign", "ridge_stats",
                                                 "ridge_apply") if reg[r]["launches_per_step"] > 0}
    total_ms = sum(reg[r]["ms_per_step"] for r in ("update_R", "assign", "plan", "ridge_stats", "ridge_solve",
                                                   "ridge_apply"))
    kernels = {}
    for r, ms_r in timed.items():
        # kernel-named regions (k_*) wrap exactly one kernel per launch; the others wrap the hot kernel plus a
        # tiny finalize launch, so the region time itself is the (upper bound of the) kernel time
        n_launch = reg[r]["launches_per_step"] if r.startswith("k_") else 1.0
        t_launch = ms_r / n_launch * 1e-3
        ach = algo[r] * n_local / t_launch / 1e9
        kernels[r] = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                      "frac": ach / peaks["hbm_gbs"], "algorithmic_bytes_per_launch": algo[r] * n_local,
                      "avg_launch_us": t_launch * 1e6, "launches_per_step": n_launch,
                      "share_of_step": ms_r / max(1e-9, total_ms)}
    roofline = None
    if kernels:
        top = max(kernels, key=lambda r: kernels[r]["share_of_step"])
        # DRAM bytes of one launch of the dominant kernel from the ncu --set full capture of this exact
        # workload (profiles/r01_final_kernels.md: dram__bytes_read.sum + dram__bytes_write.sum); null otherwise
        traffic = measured_traffic(top, args.config, n_local)
        roofline = dict(kernel=top, traffic=traffic, peak_kind=peak_kind, **kernels[top])
    step_ach = ALGO_BYTES_PER_CELL_ITER * n_local / (ms_per_step * 1e-3) / 1e9

    # ---- e2e: public API with host buffers (pinned), H2D of inputs and D2H of the result in the timed region
    e2e = None
    if not args.no_e2e:
        del g
        iters_e2e = 10                                  # RunHarmony's default max_iter (R/ui.R:98)
        Zp = torch.from_numpy(Z).pin_memory().numpy()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g2 = harmony(device=local_rank, comm=new_comm())
        g2.setup(Zp, kw["phi"], kw["sigma"], kw["theta"], None, kw["alpha"], T, 1e-3, -np.inf, K, 0.05, kw["B_vec"],
                 kw["cutoff"])
        g2.set_seed(1234)
        g2.init_cluster_cpp()                            # native kmeans_centers (utils.cpp:10-64), like RunHarmony()
        for _ in range(iters_e2e):
            step(g2)
        out = g2.getZcorr()
        g2.synchronize()
        t_e2e = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([t_e2e], device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_e2e = float(tt.item())
        assert np.all(np.isfinite(out[:, :8]))
        e2e = {"value": N_global * iters_e2e / t_e2e, "unit": "cells/s/iter",
               "h2d_bytes_per_step": int((Z.nbytes + kw["phi"].nbytes) * world / iters_e2e),
               "d2h_bytes_per_step": int(out.nbytes * world / iters_e2e),
               "iterations": iters_e2e, "seconds": t_e2e,
               "what": "harmony() + setup (H2D, pinned host Z fp64) + init_cluster_cpp with the NATIVE k-means "
                       "initialisation + 10 x harmonize body + getZcorr (D2H fp64); bytes are per iteration (totals / 10)"}
        del g2

    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_sample = cpu_sample_cells()
        t_iter, blas = cpu_reference_run(n_sample, 2, 1)
        cpu = {"value": n_sample / t_iter, "unit": "cells/s/iter", "cores": 1, "kind": "port",
               "sample": f"{n_sample} cells x {D} PCs, K={K}, levels {W['B_vec']}, 2 timed iterations, single thread "
                         f"(reference default ncores=1), sgemm from {os.path.basename(blas)}"}
        # a bounded sample through the GPU path, held against the oracle (the oracle as the checker)
        parity = parity_on_sample(local_rank, n_cells=min(50_000, n_sample))

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "cells/s/iter", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"synthetic {N_global} cells x {D} PCs, {len(W['B_vec'])} covariate(s) (levels "
                                       f"{W['B_vec']}), K={K}, T={T}, block_size=0.05 ({W['name']})",
                           "config_id": args.config,
                           "cells_per_gpu": n_local, "parallelism": f"cells sharded x{world}",
                           "switches": sorted(k for k in os.environ if k.startswith("HB_")) + ([f"kernel_set={args.kernel_set}"] if args.kernel_set else []),
                           "l2": f"state (U,R,Z = {n_local * (2 * KS + 2 * DS) * 4 / 1e9:.1f} GB per GPU) is far larger than the 126 MB L2"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
                "roofline": roofline,
                "roofline_kernels": {r: {k2: (round(v2, 4) if isinstance(v2, float) else v2) for k2, v2 in kv.items()}
                                     for r, kv in kernels.items()},
                "roofline_step": {"bound": "hbm", "achieved": step_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                  "frac": step_ach / peaks["hbm_gbs"],
                                  "algorithmic_bytes_per_cell_iter": ALGO_BYTES_PER_CELL_ITER},
                "regions_ms_per_step": {r: round(v["ms_per_step"], 4) for r, v in reg.items()},
                "cpu_baseline": cpu, "parity": parity}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
