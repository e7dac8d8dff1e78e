#!/usr/bin/env python
"""End to end on BASELINE.json config 3 (1M cells x 50 PCs, 20 batches, K=100) through the two ways into and out of
the library, in one process on one GPU:

  host    what bench.py's `e2e` times: harmony() + setup from pinned host fp64 Z + the native k-means initialisation
          + 10 harmonize() bodies + getZcorr() (D2H, widened to fp64)
  tensor  the same with the inputs already on the device: setup from a CUDA fp32 tensor (the generator's values are
          fp32, so both paths see the same numbers) and an int32 CUDA tensor of level rows, output through
          to_torch("Z_corr") (a CUDA fp32 tensor)

Every clock read follows a device synchronise.  Both paths are warmed up, then run alternately; the JSON line has the
median / min / max of each, the HB_TRACE_HOST phases of one extra traced run of each, the rel-L2 between the two
outputs and the GPU's name and power limit.

    python scripts/bench_device_io.py [--runs 7] [--out FILE]
"""
import argparse
import contextlib
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (config 3 inputs: synth_shard / setup_kwargs)

ITERS = 10   # RunHarmony's default max_iter (R/ui.R:98), as bench.py's e2e


def gpu_card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # nvidia-smi missing: the name from torch, power limit unknown
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": None, "note": repr(e)}


@contextlib.contextmanager
def captured_stderr(sink):
    """fd-level capture of stderr (the library's HB_TRACE_HOST lines come from C)."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            yield
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
            f.seek(0)
            sink.append(f.read())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=7, help="timed runs of each path (alternating)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    from harmony_b200.harmony import harmony
    if not torch.cuda.is_available():
        raise SystemExit("bench_device_io.py needs a CUDA device")
    torch.cuda.set_device(0)
    W, T = bench.W, bench.T
    K = W["K"]
    Z, lv = bench.synth_shard(W["cells_per_gpu"], 0, 20260922 + 3)
    kw = bench.setup_kwargs(lv)
    Zp = torch.from_numpy(Z).pin_memory().numpy()
    Zt = torch.from_numpy(Z).to(device="cuda", dtype=torch.float32)
    assert torch.equal(Zt.double().cpu(), torch.from_numpy(Z))          # fp32 values: both paths see the same numbers
    phi_t = torch.from_numpy(kw["phi"]).cuda()
    setup_rest = (kw["sigma"], kw["theta"], None, kw["alpha"], T, 1e-3, -np.inf, K, 0.05, kw["B_vec"], kw["cutoff"])

    def run(path):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g = harmony(device=0)
        g.setup(Zp if path == "host" else Zt, kw["phi"] if path == "host" else phi_t, *setup_rest)
        g.set_seed(1234)
        g.init_cluster_cpp()
        for _ in range(ITERS):
            assert g.cluster_cpp() == 0
            g.moe_correct_ridge_cpp()
            g.check_convergence(1)
        out = g.getZcorr() if path == "host" else g.to_torch("Z_corr")
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    for path in ("host", "tensor"):                                     # warm-up
        run(path)
    times = {"host": [], "tensor": []}
    outs = {}
    for _ in range(args.runs):
        for path in ("host", "tensor"):
            t, outs[path] = run(path)
            times[path].append(t * 1e3)
    host_out = outs["host"].T
    dev_out = outs["tensor"].double().cpu().numpy()
    parity = float(np.linalg.norm(dev_out - host_out) / np.linalg.norm(host_out))

    traces = {}
    os.environ["HB_TRACE_HOST"] = "1"
    for path in ("host", "tensor"):
        sink = []
        with captured_stderr(sink):
            run(path)
        traces[path] = [{"call": m.group(1), "phase": m.group(2).strip(), "ms": float(m.group(3))}
                        for m in re.finditer(r"\[hb\] (\S+): (.+?)\s+([0-9.]+) ms", sink[0])]
    del os.environ["HB_TRACE_HOST"]

    def stats(v):
        return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)),
                "runs_ms": [round(x, 3) for x in v]}

    line = {"what": "end to end, config 3: harmony() + setup + native k-means init + 10 harmonize() bodies + Z_corr out",
            "workload": f"synth_shard {W['cells_per_gpu']} cells x {W['d']} PCs, levels {W['B_vec']}, K={K}, T={T}, "
                        f"block_size=0.05 (BASELINE.json config 3)",
            "gpu": gpu_card(), "iterations": ITERS, "warmup_runs_per_path": 1,
            "host": dict(stats(times["host"]), inputs="pinned host fp64 Z + int32 phi", output="getZcorr() fp64 host"),
            "tensor": dict(stats(times["tensor"]), inputs="CUDA fp32 Z + CUDA int32 phi", output="to_torch() fp32 CUDA"),
            "speedup_median": float(np.median(times["host"]) / np.median(times["tensor"])),
            "parity_rel_l2_zcorr": parity,
            "host_trace_ms": traces}
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
